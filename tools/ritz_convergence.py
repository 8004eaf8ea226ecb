"""Convergence of Deep Ritz with Neumann / Robin data on one GPU, in the Ritz form and the penalty form of the boundary
term (prints one JSON object; ``--out FILE`` also writes it there, default profiles/ritz_convergence.json).

-Lap u = f on [0, 2]^2 with the manufactured solution u* = sin(k_0 pi x_0 / 2) sin(k_1 pi x_1 / 2), ks = (1, 1.5), so
that u* is not 0 on the hi face of axis 1.  An 'RB' SolutionNet [2, 64, 64, 64, 64, 1] (sin, float32) is trained by the
graphed FusedTrainer (method 'DRM', 20 000 fixed interior points, 4000 fresh face points per epoch, Adam lr 1e-3):

  (a) Robin du/dn + u = g on every face (robin_kappa = 1);
  (b) Neumann du/dn = g on the axis-1 faces, the soft Dirichlet penalty (weight 1e4) on the axis-0 faces;
  (c) pure Neumann on every face, with the mean constraint (mean_value=True).

Each case runs with neumann_form='ritz' (the boundary term of the functional, PROG_RITZ_VALUE) and 'penalty'
(mean((du/dn + kappa u - g)^2), PROG_FLUX, weight 1).  Recorded per run: the L2 error against u* on 4000 fresh test
points at every checkpoint, the best L2 error seen, and the time per graphed epoch (CUDA events around the replays
between checkpoints), with the device name and power limit.

    python tools/ritz_convergence.py [--epochs 4000] [--every 250] [--out FILE]
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

L_BOX, KS = 2.0, [1.0, 1.5]
CASES = {
    "a": dict(neumann_faces=0b1111, robin_kappa=1.0),
    "b": dict(neumann_faces=0b1100),
    "c": dict(neumann_faces=0b1111, mean_value=True),
}


def device():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def run_case(case, form, epochs, every=None, seed=0):
    """(final L2 error, record) of one graphed training run of case ``case`` in ``form`` ('ritz' | 'penalty')."""
    every = every or epochs
    torch.manual_seed(seed)
    model = pb.poisson.SolutionNet(2, 64, 5, "RB").cuda()
    tr = pb.train.FusedTrainer(model, L_BOX, KS, method="DRM", n_interior=20000, n_boundary=4000, lr=1e-3, seed=seed,
                               n_test=4000, neumann_form=form, graph=True, **CASES[case])
    l2, ms, done = [], [], 0
    while done < epochs:
        k = min(every, epochs - done)
        if done == 0:          # the first epoch runs eagerly and captures the graph: not timed
            tr.step(1)
            done, k = 1, k - 1
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tr.step(k)
        b.record()
        torch.cuda.synchronize()
        if k:
            ms.append((k, a.elapsed_time(b)))
        done += k
        l2.append([done, float(tr.l2)])
    n_timed = sum(k for k, _ in ms)
    rec = {"case": case, "form": form, "rows": tr.rows, "weights": {t: tr.w[t] for t in tr.rows},
           "l2": l2, "best_l2": float(tr.best_l2), "ms_per_epoch": sum(t for _, t in ms) / max(n_timed, 1),
           "terms": {k: float(v) for k, v in tr.terms.items()}}
    return l2[-1][1], rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=4000)
    ap.add_argument("--every", type=int, default=250)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ritz_convergence.json"))
    args = ap.parse_args()
    out = {"device": device(), "problem": {"dim": 2, "L": L_BOX, "ks": KS, "model": "SolutionNet(2, 64, 5, 'RB') fp32",
                                           "method": "DRM", "n_interior": 20000, "n_boundary": 4000, "n_test": 4000,
                                           "lr": 1e-3, "seed": 0, "epochs": args.epochs},
           "runs": []}
    for case in CASES:
        for form in ("ritz", "penalty"):
            out["runs"].append(run_case(case, form, args.epochs, args.every)[1])
    s = json.dumps(out)
    print(s)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
