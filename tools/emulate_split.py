"""CPU emulation of the tensor-core operand splits (development aid): rounds GEMM operands the way
the tcgen05 path does (x = hi + lo in bf16 / fp16, fp32 accumulate) inside the forward / dgrad /
wgrad contractions of the 3-D PINN step and reports loss / gradient error vs float64.

Box-size sweep: W0 is multiplied by 2 / L and the points are drawn in [0, L)^3, so the pre-activations are the same at
every L while the derivative channels scale with 2 / L.  `rescale` runs the kernel's first-layer coordinates x' = 2^-K x,
W0' = 2^K W0 (K = -round(log2 max|W0|) outside max|W0| in [2^-2, 2^2], pde_tc.cu); `split_xt` also splits the x^T
operand of the first-layer gradient."""
import sys, os, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from oracle import jets_numpy as O

def split(x, fmt, terms):
    t = torch.from_numpy(x.astype(np.float32))
    dt = torch.bfloat16 if fmt == "bf16" else torch.float16
    hi = t.to(dt).float()
    if terms == 1:
        return [hi.numpy().astype(np.float64)]
    lo = (t - hi).to(dt).float()
    return [hi.numpy().astype(np.float64), lo.numpy().astype(np.float64)]

def mm(a, b, fmt, mode):
    """a @ b with split operands. mode: 'fp32' exact, '1', '3' (hh+hl+lh), '4'."""
    if mode == "fp32":
        return (a.astype(np.float32) @ b.astype(np.float32)).astype(np.float64)
    A = split(a, fmt, 1 if mode == "1" else 2); B = split(b, fmt, 1 if mode == "1" else 2)
    out = A[0] @ B[0]
    if mode in ("3", "4"):
        out = out + A[0] @ B[1] + A[1] @ B[0]
    if mode == "4":
        out = out + A[1] @ B[1]
    return out.astype(np.float32).astype(np.float64)

def kernel_k(W0):
    m = np.abs(W0).max()
    return 0 if 0.25 <= m <= 4 else -round(math.log2(m))

def run(fmt, mode, N=4096, d=3, seed=0, L=2.0, rescale=False, split_xt=False):
    rng = np.random.default_rng(seed)
    torch.manual_seed(seed)
    import pde_b200  # noqa
    from pde_b200.poisson import SolutionNet, rhs_f_for_u_sin
    m = SolutionNet(d, 64, 5, "RB")
    lin = [x for x in m.net if isinstance(x, torch.nn.Linear)]
    Ws = [l.weight.detach().double().numpy() for l in lin]; bs = [l.bias.detach().double().numpy() for l in lin]
    Ws[0] = Ws[0] * (2.0 / L)
    X = rng.uniform(0, L, (N, d)); f = rhs_f_for_u_sin(torch.tensor(X), L, [1] * d).numpy()
    ref_loss, rW, rb = O.poisson_pinn_loss(Ws, bs, X, f, L, "RB")
    # emulated: same algorithm, hidden GEMMs through mm(), in the coordinates x' = X / sc with seeds sc W0
    C = 1 + 2 * d; n = len(Ws)
    sc = 2.0 ** (kernel_k(Ws[0]) if rescale else 0)
    Xs = X / sc
    a = [X] + [np.broadcast_to(np.eye(d)[i] * sc, (N, d)) for i in range(d)] + [np.zeros((N, d)) for _ in range(d)]
    Zs = []; As = []
    for l in range(n - 1):
        W, b = Ws[l], bs[l]
        if l == 0:
            z = [ai @ W.T for ai in a]
        else:
            z = [mm(ai, W.T, fmt, mode) for ai in a]
        z[0] = z[0] + b
        Zs.append(z); As.append(a)
        s0, s1, s2, s3 = O._act(z[0], O.SIN)
        a = [s0] + [s1 * z[1 + i] for i in range(d)] + [s2 * z[1 + i] ** 2 + s1 * z[1 + d + i] for i in range(d)]
        a = [x.astype(np.float32).astype(np.float64) for x in a]
    J = np.concatenate([ai @ Ws[-1].T + (bs[-1] if k == 0 else 0) for k, ai in enumerate(a)], axis=1)
    J[:, 1:1 + d] /= sc; J[:, 1 + d:] /= sc * sc
    U, ctx = O.apply_envelope(J, X, 2, O.ENV_NONE, 0.0, L)
    q, Ub, _ = O.pinn_program(U, d, f, alpha=-1.0)
    loss = q.mean()
    Jb = O.envelope_backward(Ub / N, ctx, 2, d)
    Jb[:, 1:1 + d] /= sc; Jb[:, 1 + d:] /= sc * sc
    bscale = 2.0 ** (1 - np.floor(np.log2(np.abs(Jb).max())))   # the kernel's adjoint scale: largest cotangent in [2, 4)
    Jb = Jb * bscale
    gW = [None] * n; gb = [None] * n
    zb = [Jb[:, c:c + 1] for c in range(C)]
    gW[-1] = sum(zb[c].T @ a[c] for c in range(C)); gb[-1] = zb[0].sum(0)
    ab = [zb[c] @ Ws[-1] for c in range(C)]
    for l in range(n - 2, -1, -1):
        z = Zs[l]
        s0, s1, s2, s3 = O._act(z[0], O.SIN)
        nz = [None] * C
        nz[0] = s1 * ab[0]
        for i in range(d):
            nz[0] = nz[0] + s2 * z[1 + i] * ab[1 + i] + (s3 * z[1 + i] ** 2 + s2 * z[1 + d + i]) * ab[1 + d + i]
            nz[1 + i] = s1 * ab[1 + i] + 2 * s2 * z[1 + i] * ab[1 + d + i]
            nz[1 + d + i] = s1 * ab[1 + d + i]
        nz = [x.astype(np.float32).astype(np.float64) for x in nz]
        ain = As[l]
        if l == 0:
            xt = mm(nz[0].T, Xs, fmt, mode) if split_xt else nz[0].T @ Xs
            gW[0] = (xt + sum(nz[c].T @ ain[c] / sc for c in range(1, C))) * sc
        else:
            gW[l] = sum(mm(nz[c].T, ain[c], fmt, mode) for c in range(C))
            ab = [mm(nz[c], Ws[l], fmt, mode) for c in range(C)]
        gb[l] = nz[0].sum(0)
    gW = [g / bscale for g in gW]; gb = [g / bscale for g in gb]
    per = max(np.linalg.norm(a - b) / np.linalg.norm(b) for a, b in zip(gW + gb, rW + rb) if np.linalg.norm(b) > 0)
    return abs(loss - ref_loss) / abs(ref_loss), per

if __name__ == "__main__":
    # worst per-tensor gradient error (relative L2) vs float64 over the box-size sweep
    boxes = [2.0 / 64, 2.0, 8.0, 20.0, 60.0, 200.0, 2000.0]
    print(f"{'box side L':<28}" + "".join(f"{L:>10.4g}" for L in boxes))
    for label, kw in [("fp16x3", {}), ("fp16x3, x^T split", {"split_xt": True}),
                      ("fp16x3, rescaled", {"rescale": True}), ("fp16x3, rescaled, x^T split", {"rescale": True, "split_xt": True}),
                      ("fp32 GEMMs", {"fmt": "fp16", "mode": "fp32"})]:
        fmt, mode = kw.pop("fmt", "fp16"), kw.pop("mode", "3")
        res = [run(fmt, mode, L=L, **kw) for L in boxes]
        print(f"{label:<28}" + "".join(f"{g:>10.1e}" for _, g in res) + f"   (loss: worst {max(l for l, _ in res):.1e})")
