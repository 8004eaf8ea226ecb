import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    """A fixture's arrays; large weights stored as float32 (exact, make_golden.shrink) come back as float64."""
    with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
        return {k: z[k].astype(np.float64) if z[k].dtype == np.float32 and not k.startswith("ref32_") else z[k]
                for k in z.files}


def net_from(g, prefix=""):
    Ws, bs = [], []
    i = 0
    while f"{prefix}W{i}" in g:
        Ws.append(g[f"{prefix}W{i}"]); bs.append(g[f"{prefix}b{i}"]); i += 1
    return Ws, bs


def grads_from(g, prefix=""):
    gWs, gbs = [], []
    i = 0
    while f"{prefix}gW{i}" in g:
        gWs.append(g[f"{prefix}gW{i}"]); gbs.append(g[f"{prefix}gb{i}"]); i += 1
    return gWs, gbs


def stored_entries(got, g, prefix=""):
    """Full gradients (gW, gb) reduced to what fixture g stores for `prefix`: a large tensor is stored as a fixed
    sample of its entries, with their flat indices in <key>_idx (make_golden.shrink)."""
    def pick(a, key):
        return np.asarray(a).reshape(-1)[g[key + "_idx"]] if key + "_idx" in g else a
    gW, gb = got
    return ([pick(a, f"{prefix}gW{i}") for i, a in enumerate(gW)], [pick(a, f"{prefix}gb{i}") for i, a in enumerate(gb)])


def flat(gWs, gbs):
    """Flatten in nn.Module.parameters() order: W0, b0, W1, b1, ..."""
    return np.concatenate([np.concatenate([np.asarray(W).reshape(-1), np.asarray(b).reshape(-1)]) for W, b in zip(gWs, gbs)])


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    den = np.linalg.norm(b)
    return np.linalg.norm(a - b) / (den if den > 0 else 1.0)


def rel_max(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    den = np.max(np.abs(b))
    return np.max(np.abs(a - b)) / (den if den > 0 else 1.0)


def grads_err(got, want):
    """Largest relative error by the two gradient criteria of SURVEY.md §8d: per-parameter-tensor relative L2
    (for tensors that carry signal) and max-abs over the largest gradient entry.  Returns (error, where)."""
    (gW, gb), (wW, wb) = got, want
    scale = max(max(np.max(np.abs(w)) for w in wW), max(np.max(np.abs(b)) for b in wb))
    scale = scale if scale > 0 else 1.0
    worst, where = 0.0, ""
    for i, (a, b) in enumerate(zip(list(gW) + list(gb), list(wW) + list(wb))):
        b = np.asarray(b, dtype=np.float64)
        a = np.asarray(a, dtype=np.float64).reshape(b.shape)
        nb = np.linalg.norm(b)
        if nb > 1e-3 * scale * np.sqrt(b.size):
            e = np.linalg.norm(a - b) / nb
            if not e <= worst:
                worst, where = e, f"tensor {i} rel l2"
        e = np.max(np.abs(a - b)) / scale
        if not e <= worst:
            worst, where = e, f"tensor {i} max abs"
    return worst, where


def _log(kind, what, err, tol):
    """PDE_PARITY_LOG=<file>: every parity comparison (measured error, bar) is appended to it — the table under
    profiles/ is made this way."""
    path = os.environ.get("PDE_PARITY_LOG")
    if path:
        test = os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0]
        with open(path, "a") as fh:
            fh.write(f"{test}\t{kind}\t{what.strip()}\t{err:.3e}\t{tol:.3e}\n")


def assert_grads_close(got, want, tol, what=""):
    """Per-parameter-tensor relative L2 and global max-abs criteria (SURVEY.md §8d)."""
    e, where = grads_err(got, want)
    _log("grad", what, e, tol)
    assert e <= tol, f"{what} {where}: {e:.3e} > {tol:.3e}"


# ---- parity bars.  north_star: 1e-5 relative in fp32, 1e-10 in fp64, against the reference's float64 outputs.
# A float32 bar may be raised ONLY to twice the distance between the reference's own float32 run and its
# float64 run (make_golden.py stores it as e32_*: the worst case over the fixture and eight inputs one float32 ulp
# away, because a single draw of a cancelling quantity is not representative): where the reference's fp32
# arithmetic is itself further than 5e-6 from its fp64 result, no fp32 implementation can be asked to do better.
# float64 bars are never raised: the stored conditioning figures (c64_*, <= 3e-14 on every fixture) show that a
# 1-ulp change of the inputs moves no output by more than 3e-14 relative.
BASE_TOL = {"float32": 1e-5, "float64": 1e-10}


def _dt(dtype):
    return str(dtype).replace("torch.", "")


def loss_bar(g, key, dtype):
    base = BASE_TOL[_dt(dtype)]
    if _dt(dtype) == "float64" or ("e32_" + key) not in g:
        return base
    return max(base, 2.0 * float(g["e32_" + key][0]) / max(abs(float(g[key])), 1e-3))


def grads_bar(g, prefix, dtype):
    """Same two criteria as grads_err, evaluated on the reference's own float32 error of each tensor."""
    base = BASE_TOL[_dt(dtype)]
    if _dt(dtype) == "float64" or ("e32_" + prefix + "gW0") not in g:
        return base
    wW, wb = grads_from(g, prefix)
    names = [f"{prefix}gW{i}" for i in range(len(wW))] + [f"{prefix}gb{i}" for i in range(len(wb))]
    scale = max(max(np.max(np.abs(w)) for w in wW), max(np.max(np.abs(b)) for b in wb))
    scale = scale if scale > 0 else 1.0
    worst = 0.0
    for nm, b in zip(names, list(wW) + list(wb)):
        emax, el2 = (float(v) for v in g["e32_" + nm])
        nb = np.linalg.norm(b)
        if nb > 1e-3 * scale * np.sqrt(b.size):
            worst = max(worst, el2 / nb)
        worst = max(worst, emax / scale)
    return max(base, 2.0 * worst)


def assert_loss_close(got, g, key, dtype, what=""):
    got = float(got.detach()) if hasattr(got, "detach") else float(got)
    want, tol = float(g[key]), loss_bar(g, key, dtype)
    e = abs(got - want) / max(abs(want), 1e-3)
    _log("loss", f"{what} {key}", e, tol)
    assert e <= tol, f"{what} {key}: {got!r} vs {want!r}: {e:.3e} > {tol:.3e}"


def assert_grads_golden(got, g, prefix, dtype, what=""):
    assert_grads_close(stored_entries(got, g, prefix), grads_from(g, prefix), grads_bar(g, prefix, dtype), f"{what} {prefix}")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
