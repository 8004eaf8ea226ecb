"""Time of one heat-equation loss step (forward + parameter gradient) three ways, on the same network and points
(prints one JSON object; ``--out FILE`` also writes it there, default profiles/heat_time.json).

Network [4, 64, 64, 64, 64, 1] sin, float32 (3-D space + time), 2^22 points in [0, 1]^4, kappa = 0.1, f given:

  parabolic  one fused PROG_PARABOLIC call (heat.heat_residual_loss) + backward;
  pinn       one fused PROG_PINN call (alpha = -kappa) on the same network and points + backward: the stationary
             program with the same channel count, for comparison;
  composed   ops.mlp_jets(order=2) (value, gradient and Hessian diagonal written to HBM), the residual
             u_t - kappa Lap_x u - f in torch ops, and autograd back through pde_jets_backward.

Every variant is warmed up, then the variants are alternated for ``--rounds`` rounds of ``--steps`` steps each, timed
with CUDA events around each window (median and spread over the rounds).  The parabolic and composed losses and
gradients are compared on the same inputs.  Device name and power limit are recorded with the numbers.

    python tools/heat_time.py [--points 4194304] [--steps 5] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pde_b200 as pb  # noqa: E402
from pde_b200 import _lib as L  # noqa: E402
from pde_b200.ops import NO_ENVELOPE, ProgramSpec, mlp_jets, residual_mean  # noqa: E402

DIM, KAPPA = 4, 0.1


def device():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def composed_loss(model, X, f):
    """mean((u_t - kappa Lap_x u - f)^2) from the order-2 network jets and torch ops (time is the last column)."""
    J = mlp_jets(model, X, order=2)
    d = X.shape[1]
    u_t = J[:, d]                                  # channel 1 + (d - 1)
    lap = J[:, 1 + d:1 + 2 * d - 1].sum(dim=1)     # Hessian diagonal of the spatial columns
    r = u_t - KAPPA * lap - f
    return (r * r).mean()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=1 << 22)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "heat_time.json"))
    args = ap.parse_args()
    torch.manual_seed(0)
    model = pb.poisson.SolutionNet(DIM, 64, 5, "RB").cuda()
    X = torch.rand(args.points, DIM, device="cuda")
    f = torch.cos(X).sum(dim=1)
    params = list(model.parameters())
    variants = {
        "parabolic": lambda: pb.heat.heat_residual_loss(model, X, f, KAPPA),
        "pinn": lambda: residual_mean(model, X, ProgramSpec(L.PROG_PINN, alpha=-KAPPA), NO_ENVELOPE, f=f),
        "composed": lambda: composed_loss(model, X, f),
    }
    family, launches = {}, {}

    def step(name):
        for p in params:
            p.grad = None
        loss = variants[name]()
        loss.backward()
        return loss

    values = {}
    for name in variants:      # warm-up, kernel family, launches per step, and the values compared below
        for _ in range(3):
            step(name)
        torch.cuda.synchronize()
        c0 = pb.ops.launch_count()
        loss = step(name)
        torch.cuda.synchronize()
        launches[name] = pb.ops.launch_count() - c0
        family[name] = pb.ops.last_kernel_path()
        values[name] = (float(loss.detach()), torch.cat([p.grad.reshape(-1) for p in params]).double())

    times = {name: [] for name in variants}
    for _ in range(args.rounds):
        for name in variants:
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.steps):
                step(name)
            b.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(b) / args.steps)

    lp, gp = values["parabolic"]
    lc, gc = values["composed"]
    out = {"device": device(),
           "problem": {"net": "SolutionNet(4, 64, 5, 'RB') sin fp32", "points": args.points, "kappa": KAPPA,
                       "steps_per_window": args.steps, "rounds": args.rounds, "timing": "CUDA events, variants alternated"},
           "ms_per_step": {k: statistics.median(v) for k, v in times.items()},
           "ms_per_step_all": times,
           "kernel_path": family,
           "library_launches_per_step": launches,
           "parabolic_vs_composed": {"loss_rel": abs(lp - lc) / abs(lc),
                                     "grad_rel_l2": float(torch.linalg.norm(gp - gc) / torch.linalg.norm(gc))}}
    med = out["ms_per_step"]
    out["ratios"] = {"composed_over_parabolic": med["composed"] / med["parabolic"],
                     "parabolic_over_pinn": med["parabolic"] / med["pinn"]}
    s = json.dumps(out)
    print(s)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
