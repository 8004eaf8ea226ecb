"""Convergence of the heat equation on the fused path on one GPU (prints one JSON object; ``--out FILE`` also writes it
there, default profiles/heat_convergence.json).

u_t = kappa Lap_x u on [0, 1]^2 x [0, 1] (2-D space, then time), kappa = 0.1, with the exact solution
u* = exp(-kappa lambda t) sin(pi x_0) sin(pi x_1) (pde_b200.heat.exact_u_heat, ks = (1, 1)).  An 'RB' SolutionNet
[3, 64, 64, 64, 64, 1] (sin, float32) is trained with pb.train.Adam (lr 1e-3) inside one pb.train.GraphedEpoch:

  - residual: heat_residual_loss with f = 0 on 2^16 fresh interior points per epoch (PROG_PARABOLIC, tensor cores);
  - initial penalty: poisson.data_loss against u*(x, 0) on 4096 fresh points of heat.initial_face(3), weight 10;
  - Dirichlet penalty: mean(u^2) (PROG_MSE) on 4 x 1024 fresh points of heat.spatial_faces(3), weight 10.

All points come from the device samplers with the Adam step counter as the Philox offset, so every replay draws fresh
points.  Recorded: the relative L2 error against u* on 2^16 fixed test points at every checkpoint, the best one seen,
the time per graphed epoch (CUDA events around the replays between checkpoints), the kernel family of the residual,
and the device name and power limit.

    python tools/heat_convergence.py [--epochs 6000] [--every 500] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pde_b200 as pb  # noqa: E402
from pde_b200 import _lib as L  # noqa: E402
from pde_b200.ops import NO_ENVELOPE, ProgramSpec  # noqa: E402

DIM, L_BOX, KS, KAPPA = 3, 1.0, [1, 1], 0.1
N_INTERIOR, N_FACE, N_TEST = 1 << 16, 4096, 1 << 16
W_INIT, W_BC, LR = 10.0, 10.0, 1e-3


def device():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def run(epochs, every=None, seed=0):
    """(final relative L2 error, record) of one graphed training run."""
    every = every or epochs
    torch.manual_seed(seed)
    model = pb.poisson.SolutionNet(DIM, 64, 5, "RB").cuda()
    opt = pb.train.Adam(model.parameters(), lr=LR)
    step = opt.state["step"]
    X = torch.empty(N_INTERIOR, DIM, device="cuda")
    X0 = torch.empty(N_FACE, DIM, device="cuda")
    sf = pb.heat.spatial_faces(DIM)
    Xb = torch.empty(bin(sf).count("1") * (N_FACE // 4), DIM, device="cuda")
    family = {}

    def epoch():
        opt.zero_grad()
        pb.train.sample_points_rhs(N_INTERIOR, DIM, L_BOX, seed=seed, offset_add=step, out=(X, None, None))
        pb.train.sample_faces_rhs(N_FACE, DIM, L_BOX, faces=pb.heat.initial_face(DIM), seed=seed + 1, offset_add=step,
                                  out=(X0, None))
        pb.train.sample_faces_rhs(N_FACE // 4, DIM, L_BOX, faces=sf, seed=seed + 2, offset_add=step, out=(Xb, None))
        res = pb.heat.heat_residual_loss(model, X, None, KAPPA)
        family.setdefault("residual", pb.ops.last_kernel_path())
        init = pb.poisson.data_loss(model, X0, pb.heat.exact_u_heat(X0, L_BOX, KS, KAPPA), L_BOX)
        bc = pb.ops.residual_mean(model, Xb, ProgramSpec(L.PROG_MSE), NO_ENVELOPE)
        loss = res + W_INIT * init + W_BC * bc
        loss.backward()
        opt.step()
        return torch.stack([loss.detach(), res.detach(), init.detach(), bc.detach()])

    gen = torch.Generator(device="cuda").manual_seed(seed + 100)
    Xt = torch.rand(N_TEST, DIM, device="cuda", generator=gen) * L_BOX
    ut = pb.heat.exact_u_heat(Xt, L_BOX, KS, KAPPA)

    def rel_l2():
        with torch.no_grad():
            return float(torch.linalg.norm(model(Xt) - ut) / torch.linalg.norm(ut))

    ep = pb.train.GraphedEpoch(epoch, warmup=3)
    ep()                      # three eager epochs and the capture: not timed
    done = ep.warmup
    l2, ms = [], []
    while done < epochs:
        k = min(every - done % every, epochs - done)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            ep()
        b.record()
        torch.cuda.synchronize()
        ms.append((k, a.elapsed_time(b)))
        done += k
        l2.append([done, rel_l2()])
    n_timed = sum(k for k, _ in ms)
    terms = [float(v) for v in ep.out]
    rec = {"l2": l2, "best_l2": min(v for _, v in l2), "final_l2": l2[-1][1],
           "ms_per_epoch": sum(t for _, t in ms) / max(n_timed, 1), "kernel_path": family.get("residual"),
           "terms": dict(zip(("total", "residual", "initial", "boundary"), terms))}
    return l2[-1][1], rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=6000)
    ap.add_argument("--every", type=int, default=500)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "heat_convergence.json"))
    args = ap.parse_args()
    out = {"device": device(),
           "problem": {"dim": DIM, "time_axis": DIM - 1, "L": L_BOX, "ks": KS, "kappa": KAPPA,
                       "model": "SolutionNet(3, 64, 5, 'RB') fp32", "n_interior": N_INTERIOR, "n_initial": N_FACE,
                       "n_boundary": N_FACE, "n_test": N_TEST, "w_initial": W_INIT, "w_boundary": W_BC, "lr": LR,
                       "seed": 0, "epochs": args.epochs},
           "run": run(args.epochs, args.every)[1]}
    s = json.dumps(out)
    print(s)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
