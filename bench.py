#!/usr/bin/env python
"""bench.py — collocation points / second per train step (fwd + Laplacian + parameter gradient).

Workload (BASELINE.json configs[1]): Poisson_ND.py 3-D PINN, SolutionNet(3, 64, 5, 'FBC'),
2^22 uniform collocation points per GPU, fp32, synthetic points, random-init weights.
A "step" is what the reference does between ``opt.zero_grad()`` and ``opt.step()``:
``loss = pinn_residual_loss(model, X, f, L); loss.backward()`` (+ the gradient all-reduce when
world > 1).  Point sampling, rhs evaluation and Adam are outside the step (SURVEY.md §8d).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference            # the reference's own CPU path on the host cores
    python bench.py --dump-outputs out/         # also save the last timed step's loss and gradients as .npy

The one JSON line carries, besides the contract's keys: ``roofline`` (tensor pipe), ``cpu_baseline`` (the reference's
CPU path in the same run), ``parity`` (loss / gradient of the first 2^16 benchmarked points against the reference
algorithm in float64 on the CPU, outside the timed region), ``extra_configs`` (BASELINE configs 1, 3, 4, 5, each with its
own CPU leg) and, for N > 1, ``exchange_check`` (NVLink one-kernel exchange vs NCCL, replicas bit-identical).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

DIM, WIDTH, DEPTH, L_DOM = 3, 64, 5, 2.0
N_PER_GPU = 1 << 22
WORKLOAD = "Poisson_ND 3-D PINN FBC, SolutionNet(3,64,5) sin, 2^22 pts/GPU, fp32"
METRIC = "collocation points/sec per train step (fwd+Δu+param-grad)"
CPU_CHUNK = 1 << 16


def flop_per_point(n_hidden, H, C, d):
    """Algorithmic FLOPs per point (SURVEY.md §8d): 3 (fwd, dgrad, wgrad) x hidden GEMMs x 2 H^2 x channels + first /
    last layer terms; C = 1 + 2d (PINN), 1 + d (Deep Ritz, WAN per network)."""
    return 3 * (n_hidden - 1) * 2 * H * H * C + 6 * H * C + 4 * d * H


FLOP_PER_POINT = flop_per_point(DEPTH - 1, WIDTH, 1 + 2 * DIM, DIM)   # 519 552


def workload_config(world, points):
    """`config` of both arms: the reference arm times a bounded sample of exactly this workload."""
    return {"workload": WORKLOAD, "points_per_gpu": points, "global_points": points * world,
            "parallelism": f"dp{world} over points, one all-reduce of [grad|dE|sum] (51 KB) per step",
            "l2": "4 rotating point sets (256 MiB) > 126 MB L2"}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for nme, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# The reference's CPU path.  oracle/_ref/ holds the reference's own scripts, copied unmodified by
# __graft_entry__.build() where /root/reference exists (kind "reference"); without them the torch port of the same
# nested-autograd algorithm, oracle/autograd_ref.py, is timed instead (kind "port").
# ------------------------------------------------------------------------------------------------------------------
class PoissonCpu:
    """loss + .backward() of Poisson_ND.pinn_residual_loss / drm_energy_loss in 2^16-point chunks (one autograd graph
    of 2^22 points does not fit in host memory, SURVEY.md §5), gradients accumulating in p.grad like a training step."""

    def __init__(self, dim, bc, method, dtype=torch.float32, state=None):
        from oracle import ref_loader
        self.P = ref_loader.load("Poisson_ND.py")
        self.kind = "reference" if self.P is not None else "port"
        self.dim, self.bc, self.method, self.dtype = dim, bc, method, dtype
        if self.P is not None:
            self.model = self.P.SolutionNet(dim, WIDTH, DEPTH, bc_mode=bc).to(dtype)
            self.net = self.model.net
        else:
            from oracle import autograd_ref as AR
            self.AR = AR
            self.net = AR.build_mlp([dim] + [WIDTH] * (DEPTH - 1) + [1], "sin", dtype)
        if state is not None:      # same weights as the CUDA model (parity leg)
            lin = [m for m in self.net if isinstance(m, torch.nn.Linear)]
            with torch.no_grad():
                for m, (W, b) in zip(lin, state):
                    m.weight.copy_(W.to(dtype)); m.bias.copy_(b.to(dtype))

    def rhs(self, X):
        if self.P is not None:
            return self.P.rhs_f_for_u_sin(X, L_DOM, [1] * self.dim).detach()
        return self.AR.manufactured_rhs(X, L_DOM, [1] * self.dim)

    def step(self, X, f):
        for p in self.net.parameters():
            p.grad = None
        N, total = X.shape[0], 0.0
        for s in range(0, N, CPU_CHUNK):
            Xc = X[s:s + CPU_CHUNK].detach().clone().requires_grad_(True)
            fc = f[s:s + CPU_CHUNK]
            if self.P is not None:
                fn = self.P.pinn_residual_loss if self.method == "pinn" else self.P.drm_energy_loss
                part = fn(self.model, Xc, fc, L_DOM) * (Xc.shape[0] / N)
            else:
                fn = self.AR.pinn_loss if self.method == "pinn" else self.AR.drm_loss
                part = fn(self.net, Xc, fc, L_DOM, self.bc) * (Xc.shape[0] / N)
            part.backward()
            total += float(part.detach())
        return total

    def flat_grad(self):
        return torch.cat([p.grad.reshape(-1) for p in self.net.parameters()])

    def describe(self):
        return ("oracle/_ref/Poisson_ND.py (the reference's own file, unmodified)" if self.kind == "reference"
                else "oracle/autograd_ref.py (torch port of the reference's nested-autograd algorithm)")


def cpu_rate(leg, n_points, threads):
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    X = torch.rand(n_points, leg.dim, dtype=leg.dtype) * L_DOM
    f = leg.rhs(X)
    leg.step(X[:CPU_CHUNK], f[:CPU_CHUNK])     # warm-up
    t0 = time.perf_counter()
    leg.step(X, f)
    dt = time.perf_counter() - t0
    return n_points / dt, dt


def gpu_eager_reference_rate(dev, n_chunks=4):
    """The same nested-autograd algorithm run by PyTorch eager on the B200 itself (SURVEY.md §8d's second,
    recommended baseline): what switching the reference to `device='cuda'` gives without this library."""
    from oracle import autograd_ref as AR
    torch.manual_seed(0)
    net = AR.build_mlp([DIM] + [WIDTH] * (DEPTH - 1) + [1], "sin", torch.float32).to(dev)
    X = torch.rand(n_chunks * CPU_CHUNK, DIM, device=dev) * L_DOM
    f = AR.manufactured_rhs(X, L_DOM, [1] * DIM)
    AR.loss_and_grads("pinn", net, X[:CPU_CHUNK], f[:CPU_CHUNK], L_DOM, "FBC", chunk=CPU_CHUNK)  # warm-up
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    AR.loss_and_grads("pinn", net, X, f, L_DOM, "FBC", chunk=CPU_CHUNK)
    e1.record()
    torch.cuda.synchronize(dev)
    return X.shape[0] / (e0.elapsed_time(e1) * 1e-3)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the step on all host cores.  Each step is a bounded
    sample of the 2^22-point workload — as many 2^16-point chunks as keep the whole --steps/--warmup run near two
    minutes (the rate is per point; the reference is faster per point at 2^16 than at larger graphs, BASELINE.md §2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    leg = PoissonCpu(DIM, "FBC", "pinn")
    torch.manual_seed(0)
    X = torch.rand(N_PER_GPU, DIM) * L_DOM
    f = leg.rhs(X)
    leg.step(X[:CPU_CHUNK], f[:CPU_CHUNK])
    t0 = time.perf_counter()
    leg.step(X[:CPU_CHUNK], f[:CPU_CHUNK])
    t_chunk = time.perf_counter() - t0
    budget_s = float(os.environ.get("PDE_BENCH_REF_BUDGET_S", "120"))
    n_chunks = int(max(1, min(N_PER_GPU // CPU_CHUNK, budget_s / ((args.steps + args.warmup) * t_chunk))))
    n = n_chunks * CPU_CHUNK
    for _ in range(args.warmup):
        leg.step(X[:n], f[:n])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        leg.step(X[:n], f[:n])
    dt = time.perf_counter() - t0
    val = n * args.steps / dt
    sample = (f"{n} of the 2^22 points per step ({n_chunks} chunks of 2^16), {leg.describe()}, fp32, "
              f"{torch.get_num_threads()} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, N_PER_GPU),
        "cpu_baseline": {"value": val, "unit": "points/s", "cores": torch.get_num_threads(), "kind": leg.kind, "sample": sample},
        "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# parity of the benchmarked batch, outside the timed region
# ------------------------------------------------------------------------------------------------------------------
def parity_check(model, X, f, loss_gpu, grad_gpu, n=CPU_CHUNK):
    """Loss and gradient of the first 2^16 benchmarked points (fp32 CUDA path) against the reference algorithm in
    float64 on the CPU with the same weights."""
    lin = [m for m in model.net if isinstance(m, torch.nn.Linear)]
    state = [(m.weight.detach().double().cpu(), m.bias.detach().double().cpu()) for m in lin]
    leg = PoissonCpu(DIM, "FBC", "pinn", dtype=torch.float64, state=state)
    want = leg.step(X[:n].double().cpu(), f[:n].double().cpu())
    gw = leg.flat_grad()
    g = grad_gpu.double().cpu()
    return {"n": n, "loss_rel": abs(loss_gpu - want) / abs(want),
            "grad_rel": float((g - gw).abs().max() / gw.abs().max()),
            "grad_rel_l2": float((g - gw).norm() / gw.norm()),
            "against": leg.describe() + ", float64, same weights and points", "tolerance": 1e-5}


# ------------------------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations (N = 1 only): device-resident inputs, CUDA events, median of `reps`
# ------------------------------------------------------------------------------------------------------------------
def _timed(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def _cpu_timed(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def extra_configs(dev, peak_tflops):
    import pde_b200 as pb
    from pde_b200 import ops
    from pde_b200.schrodinger import ipw_1d_wan as W, qho_2d as Q
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    out = []

    def entry(name, n, ms, flop_pt, cpu, extra=None):
        tf = flop_pt * n / (ms * 1e-3) / 1e12
        e = {"workload": name, "points": n, "ms_per_step": ms, "us_per_step": ms * 1e3, "points_per_s": n / ms * 1e3,
             "kernel_path": ops.last_kernel_path(), "flop_per_point": flop_pt,
             "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_tflops, "unit": "TFLOP/s", "frac": tf / peak_tflops},
             "cpu_baseline": cpu}
        if extra:
            e.update(extra)
        out.append(e)

    def step(loss_fn, params):
        def run():
            for p in params:
                p.grad = None
            loss_fn().backward()
        return run

    def epochs_ms(run, inner=10, reps=10):
        """ms per whole epoch (loss step + optimiser) of a CUDA-graph-replayed epoch: what the latency-bound
        configurations get from pde_b200.train (FusedTrainer / GraphedEpoch)."""
        run(); run()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(inner):
                run()
            b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / inner)
        return statistics.median(ts)

    # configs 1 and 3: Poisson_ND on the CUDA path vs the reference's CPU path
    for name, d, n, method, bc, n_cpu in (("config 1: Poisson_ND 1-D PINN FBC, N=20000", 1, 20000, "pinn", "FBC", 20000),
                                          ("config 3: Poisson_ND 5-D Deep Ritz, raw net (natural BC), N=2^20", 5, 1 << 20, "drm", "RB", 1 << 18)):
        torch.manual_seed(0)
        m = pb.poisson.SolutionNet(d, WIDTH, DEPTH, bc).to(dev)
        X = torch.rand(n, d, device=dev) * L_DOM
        f = pb.poisson.rhs_f_for_u_sin(X, L_DOM, [1] * d)
        fn = pb.poisson.pinn_residual_loss if method == "pinn" else pb.poisson.drm_energy_loss
        ms = _timed(step(lambda: fn(m, X, f, L_DOM), list(m.parameters())))
        leg = PoissonCpu(d, bc, method)
        rate, dt = cpu_rate(leg, n_cpu, cores)
        C = 1 + 2 * d if method == "pinn" else 1 + d
        tr = pb.train.FusedTrainer(m, L_DOM, [1] * d, method=method.upper(), X=X, f=f, weights={"bc": 0.0})
        ep = epochs_ms(lambda: tr.step(), inner=10 if n <= (1 << 16) else 3)
        entry(name, n, ms, flop_per_point(DEPTH - 1, WIDTH, C, d),
              {"value": rate, "unit": "points/s", "cores": cores, "kind": leg.kind,
               "sample": f"{n_cpu} points in 2^16 chunks ({dt:.2f} s), {leg.describe()}, fp32"},
              {"fused_epoch_ms": ep, "fused_epoch_points_per_s": n / ep * 1e3,
               "fused_epoch": "loss step + fused Adam as one replayed CUDA graph (pde_b200.train.FusedTrainer)"})

    # config 4: QHO_2D eigenstate PINN residual on the 200 x 200 grid, [2,50,50,50,50,1]
    g1 = torch.linspace(-6.0, 6.0, 200)
    xg, yg = torch.meshgrid(g1, g1, indexing="ij")
    Qr = ref_loader.load("QHO_2D.py")
    for tech in ("FBC", "FN"):
        torch.manual_seed(0)
        m = Q.FCN([2, 50, 50, 50, 50, 1], 2, 1, tech).to(dev)
        xd, yd = xg.to(dev), yg.to(dev)
        E = Q.Exact_energy(2, 1, 6.0)
        ms = _timed(step(lambda: Q.PINN_loss(m, xd, yd, E, 6.0), list(m.parameters())))
        path = ops.last_kernel_path()
        if Qr is not None:
            mr = Qr.FCN([2, 50, 50, 50, 50, 1], 2, 1, tech)

            def ref_step():   # the inline residual block of train_pinn_seperate (QHO_2D.py:329-341,363-378) around the reference's FCN
                for p in mr.parameters():
                    p.grad = None
                x = xg.clone().requires_grad_(True); y = yg.clone().requires_grad_(True)
                u = mr(x, y)
                ux = torch.autograd.grad(u, x, torch.ones_like(u), create_graph=True)[0]
                uy = torch.autograd.grad(u, y, torch.ones_like(u), create_graph=True)[0]
                uxx = torch.autograd.grad(ux, x, torch.ones_like(ux), create_graph=True)[0]
                uyy = torch.autograd.grad(uy, y, torch.ones_like(uy), create_graph=True)[0]
                V = 0.5 * math.sqrt(2) ** 2 * (x ** 2 + y ** 2)
                torch.mean((-0.5 * (uxx + uyy) + V * u - E * u) ** 2).backward()
            dt = _cpu_timed(ref_step)
            cpu = {"value": 40000 / dt, "unit": "points/s", "cores": cores, "kind": "reference",
                   "sample": f"the whole 40000-point step ({dt:.2f} s): oracle/_ref/QHO_2D.py FCN + its inline residual block restated, fp32"}
        else:
            cpu = {"value": None, "unit": "points/s", "cores": cores, "kind": "port", "sample": "oracle/_ref absent: not timed"}
        ops_path = path
        optc = pb.train.Adam(m.parameters(), lr=1e-3)   # torch.optim.Adam's update in one launch, reading the loss operator's flat gradient buffer in place

        def q_epoch():
            optc.zero_grad()
            l = Q.PINN_loss(m, xd, yd, E, 6.0); l.backward(); optc.step()
            return l.detach()
        ge = pb.train.GraphedEpoch(q_epoch); ge()
        ep = epochs_ms(lambda: ge())
        entry(f"config 4: QHO_2D 2-D eigenstate PINN {tech}, [2,50,50,50,50,1], 200x200 grid", 40000, ms,
              flop_per_point(4, 50, 5, 2), cpu,
              {"kernel_path": ops_path, "fused_epoch_ms": ep, "fused_epoch_points_per_s": 40000 / ep * 1e3,
               "fused_epoch": "loss step + pde_b200.train.Adam (one-launch Adam) as one replayed CUDA graph (pde_b200.train.GraphedEpoch)"})

    # config 5: IPW_1D_WAN minimax pair, one evaluation of WAN_loss + backward into both networks
    torch.manual_seed(0)
    um = W.FCN([1, 50, 50, 50, 1], L=2.0, enforce_bc=True).to(dev)
    vm = W.FCN([1, 20, 20, 20, 1], L=2.0).to(dev)
    x = torch.linspace(0, 2, 1000, device=dev).view(-1, 1)
    ms = _timed(step(lambda: W.WAN_loss(um, vm, x, 2, 2.0)[0], list(um.parameters()) + list(vm.parameters())))
    Wr = ref_loader.load("IPW_1D_WAN.py")
    if Wr is not None:
        ur = Wr.FCN([1, 50, 50, 50, 1], num_states=2, L=2.0, enforce_bc=True)
        vr = Wr.FCN([1, 20, 20, 20, 1], num_states=2, L=2.0, enforce_bc=False)
        xc = torch.linspace(0, 2, 1000).view(-1, 1).requires_grad_(True)

        def ref_step():
            for p in list(ur.parameters()) + list(vr.parameters()):
                p.grad = None
            Wr.WAN_loss(ur, vr, xc, 2, 2.0, 1.0, 1.0)[0].backward()
        dt = _cpu_timed(ref_step, reps=10)
        cpu = {"value": 1000 / dt, "unit": "points/s", "cores": cores, "kind": "reference",
               "sample": f"the whole 1000-point evaluation ({dt * 1e3:.2f} ms): oracle/_ref/IPW_1D_WAN.py WAN_loss + backward, fp32"}
    else:
        cpu = {"value": None, "unit": "points/s", "cores": cores, "kind": "port", "sample": "oracle/_ref absent: not timed"}
    ouc = pb.train.Adam(um.parameters(), lr=1e-3)
    ovc = pb.train.Adam(vm.parameters(), lr=1e-3)

    def wan_epoch():     # IPW_1D_WAN.py:186-208: five critic steps on the frozen solution network, then one solution step
        Ju = pb.frozen_jets(um, x)
        for _ in range(5):
            ovc.zero_grad()
            W.WAN_loss(um, vm, x, 2, 2.0, u_jets=Ju)[1].backward(inputs=list(vm.parameters())); ovc.step()
        ouc.zero_grad()
        t = W.WAN_loss(um, vm, x, 2, 2.0)[0]; t.backward(inputs=list(um.parameters())); ouc.step()
        return t.detach()
    gw = pb.train.GraphedEpoch(wan_epoch); gw()
    ep = epochs_ms(lambda: gw())
    entry("config 5: IPW_1D_WAN weak residual, u [1,50,50,50,1] / v [1,20,20,20,1], N=1000 (one loss evaluation + backward)",
          1000, ms, flop_per_point(3, 50, 2, 1) + flop_per_point(3, 20, 2, 1), cpu,
          {"kernel_path": ops.last_kernel_path() + " (network jets) + wan_kernel", "note": "launch-latency bound: 1000 points",
           "fused_epoch_ms": ep, "fused_epoch_evaluations": 6,
           "fused_epoch": "the reference's minimax epoch (5 critic + 1 solution update, 6 WAN evaluations + 6 Adam steps) as one replayed CUDA graph"})
    return out


def exchange_check(model, params, X, f, group, n_global, dev):
    """One step through the one-kernel NVLink exchange and one through NCCL on the same points: the flat gradients
    agree to 1e-6 and every rank holds bit-identical values."""
    import torch.distributed as dist
    import pde_b200 as pb
    from pde_b200 import ops

    def grads():
        for p in params:
            p.grad = None
        pb.poisson.pinn_residual_loss(model, X, f, L_DOM, group=group, n_global=n_global).backward()
        return torch.cat([p.grad.reshape(-1) for p in params]).clone()
    g_nv = grads()
    saved = dict(ops._EXCHANGE)
    ops._EXCHANGE.clear()
    try:
        g_nc = grads()
    finally:
        ops._EXCHANGE.update(saved)
    rel = float((g_nv - g_nc).abs().max() / g_nc.abs().max())
    world = dist.get_world_size()
    gathered = [torch.empty_like(g_nv) for _ in range(world)]
    dist.all_gather(gathered, g_nv)
    same = all(torch.equal(gathered[0], t) for t in gathered)
    ok = torch.tensor([1.0 if (rel <= 1e-6 and same and bool(torch.isfinite(g_nv).all())) else 0.0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() != 1.0:
        raise SystemExit(f"exchange_check failed: NVLink vs NCCL rel diff {rel:.3e}, replicas identical: {same}")
    return {"status": "ok", "nvlink_vs_nccl_rel": rel, "replicas_bit_identical": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=N_PER_GPU, help="points per GPU (default 2^22, the metric's config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and parameter gradients of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs saves the outputs of --impl b200 only")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    import pde_b200 as pb
    from pde_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the collocation kernels")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    exchange = "none (one rank)"
    # stdout carries the one JSON line only: whatever libraries print while the job runs (NCCL's version banner goes to
    # stdout whatever NCCL_DEBUG_FILE says) is sent to stderr; file descriptor 1 is restored for the final print
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
        # exchange step: one kernel over NVLink peer memory (pde_allreduce_oneshot); PDE_B200_EXCHANGE=nccl keeps NCCL.
        # No fallback: if the peer buffers cannot be set up the run fails.
        if os.environ.get("PDE_B200_EXCHANGE", "nvlink") == "nvlink":
            ops.use_nvlink_exchange(None, 1 << 15, torch.float32)
            exchange = "one-kernel NVLink peer-memory all-reduce (pde_allreduce_oneshot)"
        else:
            exchange = "NCCL all-reduce"
    N = args.points
    n_global = N * world

    torch.manual_seed(0)                       # identical weights on every rank
    model = pb.poisson.SolutionNet(DIM, WIDTH, DEPTH, "FBC").to(dev)
    params = list(model.parameters())
    # 4 rotating point sets (4 x 64 MiB = 256 MiB > 126 MB L2) so that no step finds its inputs in L2
    POOL = 4
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    Xs = [torch.rand(N, DIM, device=dev, generator=gen) * L_DOM for _ in range(POOL)]
    fs = [pb.poisson.rhs_f_for_u_sin(X, L_DOM, [1] * DIM) for X in Xs]

    def step(i):
        for p in params:
            p.grad = None
        loss = pb.poisson.pinn_residual_loss(model, Xs[i % POOL], fs[i % POOL], L_DOM, group=group, n_global=n_global)
        loss.backward()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    xcheck = None
    if world > 1 and exchange.startswith("one-kernel"):
        xcheck = exchange_check(model, params, Xs[0], fs[0], group, n_global, dev)

    for i in range(args.warmup):
        step(i)
    barrier()

    # ---- timed region: device-resident inputs
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.KERNEL_EVENTS = []                     # (start, stop) CUDA events around each fused-kernel ABI call
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        loss = step(i)
    e1.record()
    barrier()
    launches = ops.launch_count() - launches0      # counted by the library at its launch sites
    kernel_path = ops.last_kernel_path()           # recorded by the library at the launch
    ms = e0.elapsed_time(e1)
    kev = ops.KERNEL_EVENTS
    ops.KERNEL_EVENTS = None
    kernel_ms = [a.elapsed_time(b) for a, b in kev]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives from its last step: the loss and every parameter's .grad (the
        # gradient is all-reduced, so rank 0 holds the global result); copied before the end-to-end steps reuse them
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        outs = {"loss": loss, **{f"grad.{n}": p.grad for n, p in model.named_parameters()}}
        for name, t in outs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.detach().float().cpu().numpy())
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = n_global * args.steps / (ms * 1e-3)

    # ---- end to end: host (pinned) inputs each step, H2D on a copy stream one step ahead, loss read back
    hX = [X.cpu().pin_memory() for X in Xs[:2]]
    hf = [f.cpu().pin_memory() for f in fs[:2]]
    dX = [torch.empty_like(Xs[0]) for _ in range(2)]
    df = [torch.empty_like(fs[0]) for _ in range(2)]
    copy_stream = torch.cuda.Stream(dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    host_loss = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]
    losses_read = []

    def upload(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[s])
            dX[s].copy_(hX[s], non_blocking=True)
            df[s].copy_(hf[s], non_blocking=True)
            ready[s].record(copy_stream)

    def e2e_steps(k):
        for s in range(2):
            freed[s].record(torch.cuda.current_stream())
        upload(0)
        for i in range(k):
            s = i % 2
            if i + 1 < k:
                upload(i + 1)
            torch.cuda.current_stream().wait_event(ready[s])
            for p in params:
                p.grad = None
            loss = pb.poisson.pinn_residual_loss(model, dX[s], df[s], L_DOM, group=group, n_global=n_global)
            loss.backward()
            freed[s].record(torch.cuda.current_stream())
            host_loss[s].copy_(loss.detach().reshape(1), non_blocking=True)
            loss_ready[s].record(torch.cuda.current_stream())
            # the caller reads every step's loss, one step late: step i is queued before the host waits for the loss
            # of step i-1, as a training loop that logs its loss would do, so the GPU does not idle on the read-back
            if i > 0:
                loss_ready[1 - s].synchronize()
                losses_read.append(float(host_loss[1 - s][0]))
        loss_ready[(k - 1) % 2].synchronize()
        losses_read.append(float(host_loss[(k - 1) % 2][0]))

    e2e_steps(2)
    losses_read.clear()
    barrier()
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    if len(losses_read) != args.steps or not all(math.isfinite(v) for v in losses_read):
        raise RuntimeError(f"end-to-end loop read {len(losses_read)} losses for {args.steps} steps: {losses_read[:4]}")
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_global * args.steps / float(t.item())
    h2d = (hX[0].numel() + hf[0].numel()) * 4

    if rank == 0:
        peaks, how = measured_peaks()
        k_ms = statistics.mean(kernel_ms) if kernel_ms else ms / args.steps
        achieved = FLOP_PER_POINT * N / (k_ms * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
                prof = json.load(fh)
        except Exception:
            pass
        cfg = workload_config(world, N)
        out = {
            "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "exchange": exchange, "kernel_path": kernel_path,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "how": "pinned host X,f -> device on a copy stream one step ahead; every step's loss is copied to pinned host memory and read by the host after the next step has been queued (all reads inside the timed region)",
                    "losses_read": len(losses_read)},
            "gpu_launches": launches,
            "gpu_launches_how": ("pde_launch_count() delta over the timed region (counted at the library's launch sites): per step "
                                 "tc_pack_kernel, tc_kernel<3,2,sin>, reduce_kernel" + (" (with the NVLink exchange in its tail)" if world > 1 else "")
                                 + "; the autograd bridge's own ATen kernels (zero-fill, scale by dLoss, view into p.grad) are not counted"),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": prof.get("dram_bytes_per_launch"),
                         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({how})",
                         "frac_of_burst_peak": achieved / float(peaks.get("bf16_tflops", peak)),
                         "kernel_ms": k_ms, "flop_per_point": FLOP_PER_POINT,
                         "tensor_pipe_active_pct_ncu": prof.get("tensor_pipe_active_pct"),
                         "traffic_source": prof.get("source"),
                         "hbm_achieved_gbs": (4 * (DIM + 1) * N) / (k_ms * 1e-3) / 1e9},
        }
        if xcheck is not None:
            out["exchange_check"] = xcheck["status"]
            out["exchange_check_detail"] = xcheck
        # parity of the benchmarked batch (first 2^16 points of point set 0), outside the timed region
        for p in params:
            p.grad = None
        n_par = min(CPU_CHUNK, N)
        lp = pb.poisson.pinn_residual_loss(model, Xs[0][:n_par], fs[0][:n_par], L_DOM)
        lp.backward()
        gflat = torch.cat([p.grad.reshape(-1) for p in params])
        par = parity_check(model, Xs[0], fs[0], float(lp.item()), gflat, n_par)
        par["kernel_path"] = ops.last_kernel_path()
        out["parity"] = par
        if par["loss_rel"] > 1e-5 or par["grad_rel"] > 1e-5:
            raise SystemExit(f"in-run parity gate failed: {par}")
        if world == 1 and not args.no_cpu_baseline:
            leg = PoissonCpu(DIM, "FBC", "pinn")
            rate, dt = cpu_rate(leg, 64 * CPU_CHUNK, os.cpu_count() or 1)
            out["cpu_baseline"] = {"value": rate, "unit": "points/s", "cores": torch.get_num_threads(), "kind": leg.kind,
                                   "sample": f"{64 * CPU_CHUNK} points = the whole 2^22-point step in 2^16 chunks ({dt:.1f} s), "
                                             f"{leg.describe()}, fp32"}
            try:
                out["torch_eager_gpu_baseline"] = {
                    "value": gpu_eager_reference_rate(dev), "unit": "points/s",
                    "sample": f"{4 * CPU_CHUNK} points in 2^16 chunks, the same nested-autograd algorithm run by PyTorch eager on this GPU, fp32"}
            except Exception as exc:      # reported extra, never fatal
                out["torch_eager_gpu_baseline"] = {"value": None, "error": type(exc).__name__}
            if not args.no_extra_configs:
                out["extra_configs"] = extra_configs(dev, peak)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
