"""Timing of the Neumann / Robin boundary term on one GPU (prints one JSON object; ``--out FILE`` also writes it there).

* the device name and power limit the numbers belong to;
* the boundary-flux program (PDE_PROG_FLUX, d = 3, [3, 64, 64, 64, 64, 1] sin, fp32, gradient included) alone, at 4000
  and 2^20 face points on four faces, on the generic SIMT kernel and on the tensor-core kernel: CUDA events around
  200 back-to-back ABI calls (pack + fused kernel + reduction each);
* the graphed FusedTrainer epoch (PINN, 'RB' model, n_boundary = 4000) at n_interior = 20 000 and 2^20, with the
  Dirichlet penalty on all six faces, and with the axis-2 faces switched to the Neumann term; library launches per
  epoch counted by pde_launch_count over one eager epoch.

    python tools/neumann_time.py [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pde_b200 as pb  # noqa: E402
from pde_b200 import _lib as L  # noqa: E402
from pde_b200.ops import NO_ENVELOPE, ProgramSpec, _Net, _ws_for  # noqa: E402

REPS = 200
MASK = 0b001111     # faces x_0 = 0, L and x_1 = 0, L


def device():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def flux_call_ms(n, path):
    torch.manual_seed(0)
    m = pb.poisson.SolutionNet(3, 64, 5, "RB").cuda()
    X, g = pb.train.sample_faces_rhs(n // 4, 3, 2.0, MASK, [1, 1, 1], seed=1)
    net = _Net(m, X)
    cnet = net.to_c(net.params)
    np_ = sum(p.numel() for p in net.params)
    row = torch.zeros(np_ + 2, device="cuda")
    prog = ProgramSpec(L.PROG_FLUX, faces=MASK).to_c(f=g)
    cenv = NO_ENVELOPE.to_c()
    lib = L.load()
    with pb.ops.kernel_path(path):
        ws = _ws_for(cnet, 1, n, X.device)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def call():
            L.check(lib.pde_residual_loss_grad(C.byref(cnet), C.byref(cenv), C.byref(prog), X.data_ptr(), n, None, 1.0 / n,
                                               row.data_ptr() + (np_ + 1) * 4, row.data_ptr(), row.data_ptr() + np_ * 4,
                                               ws.data_ptr(), ws.numel(), st), "flux")
        for _ in range(10):
            call()
        fam = lib.pde_last_kernel_path()
        before = lib.pde_launch_count()
        call()
        launches = lib.pde_launch_count() - before
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(REPS):
            call()
        b.record()
        torch.cuda.synchronize()
    return {"points": n, "path": path, "family": {0: "simt_fma", 1: "tcgen05"}.get(fam, fam),
            "launches_per_call": launches, "ms_per_call": a.elapsed_time(b) / REPS}


def epoch_ms(n_interior, neumann):
    torch.manual_seed(0)
    m = pb.poisson.SolutionNet(3, 64, 5, "RB").cuda()
    kw = dict(method="PINN", n_interior=n_interior, n_boundary=4000, seed=3,
              neumann_faces=0b110000 if neumann else None)
    lib = L.load()
    eager = pb.train.FusedTrainer(m, 2.0, [1, 1, 1], graph=False, **kw)
    eager.step(1)
    before = lib.pde_launch_count()
    eager.step(1)
    launches = lib.pde_launch_count() - before
    tr = pb.train.FusedTrainer(m, 2.0, [1, 1, 1], graph=True, **kw)
    tr.step(3)
    torch.cuda.synchronize()
    reps = REPS if n_interior <= 1 << 16 else 30
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    tr.step(reps)
    b.record()
    torch.cuda.synchronize()
    return {"n_interior": n_interior, "neumann_faces": kw["neumann_faces"], "rows": tr.rows,
            "library_launches_per_epoch": launches, "ms_per_epoch": a.elapsed_time(b) / reps, "epochs_timed": reps,
            "terms": {k: float(v) for k, v in tr.terms.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON object to this file")
    args = ap.parse_args()
    out = {"device": device(), "flux_call": [], "fused_epoch": []}
    for n in (4000, 1 << 20):
        for path in ("simt", "tc"):
            out["flux_call"].append(flux_call_ms(n, path))
    for n in (20000, 1 << 20):
        for neumann in (False, True):
            out["fused_epoch"].append(epoch_ms(n, neumann))
    s = json.dumps(out)
    print(s)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
