"""CPU tests of the host bridge in pde_b200.ops: the ctypes descriptors that ProgramSpec / WanSpec fill, the pointers
that the residual-launch helper derives from a [grad (nparam) | dE (1) | sums (K)] row, and the normalisation of the
per-call coefficients.  Tensors live on the CPU (``data_ptr()`` needs no GPU) and the launches are recorded, not run."""
import pytest
import torch

from pde_b200 import _lib as L
from pde_b200 import ops


def test_program_spec_to_c_sets_every_field():
    spec = ops.ProgramSpec(L.PROG_PINN, alpha=-0.5, beta_const=0.25, energy_const=1.5)
    f, beta, energy = torch.zeros(4), torch.zeros(4), torch.zeros(1)
    p = spec.to_c(f, beta, energy)
    assert (p.kind, p.alpha, p.beta_const, p.energy_const) == (L.PROG_PINN, -0.5, 0.25, 1.5)
    assert (p.f, p.beta, p.energy) == (f.data_ptr(), beta.data_ptr(), energy.data_ptr())
    p = spec.to_c()
    assert p.f is None and p.beta is None and p.energy is None
    assert p.kind == L.PROG_PINN and p.alpha == -0.5


def test_wan_spec_to_c_sets_every_field():
    spec = ops.WanSpec(alpha=0.5, beta_const=0.125, energy_const=2.0, w_lo=-3.0, w_hi=3.0, eps_den=1e-10)
    f, beta, energy = torch.zeros(5, dtype=torch.float64), torch.zeros(5, dtype=torch.float64), torch.zeros(1)
    w = spec.to_c(torch.float64, 2, ops.EnvelopeSpec(L.ENV_POLY, 0.0, 2.0),
                  ops.EnvelopeSpec(L.ENV_EXPWIN, -1.0, 1.0), f, beta, energy)
    assert (w.dtype, w.dim) == (L.F64, 2)
    assert (w.alpha, w.beta_const, w.energy_const, w.w_lo, w.w_hi, w.eps_den) == (0.5, 0.125, 2.0, -3.0, 3.0, 1e-10)
    assert (w.f, w.beta, w.energy) == (f.data_ptr(), beta.data_ptr(), energy.data_ptr())
    assert (w.env_u.kind, w.env_u.lo, w.env_u.hi) == (L.ENV_POLY, 0.0, 2.0)
    assert (w.env_v.kind, w.env_v.lo, w.env_v.hi) == (L.ENV_EXPWIN, -1.0, 1.0)
    w = spec.to_c(torch.float32, 1, ops.NO_ENVELOPE, ops.NO_ENVELOPE)
    assert (w.dtype, w.dim, w.env_u.kind, w.env_v.kind) == (L.F32, 1, L.ENV_NONE, L.ENV_NONE)
    assert w.f is None and w.beta is None and w.energy is None


class _Recorder:
    """Stands in for the library: records the arguments of the two residual entry points."""

    def __init__(self):
        self.calls = []

    def pde_residual_loss_grad(self, *args):
        self.calls.append(("plain", args))
        return 0

    def pde_residual_loss_grad_exchange(self, *args):
        self.calls.append(("exchange", args))
        return 0


@pytest.fixture
def recorder(monkeypatch):
    rec = _Recorder()
    monkeypatch.setattr(L, "load", lambda: rec)
    monkeypatch.setattr(ops, "_stream", lambda device: None)
    return rec


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_residual_row_pointers_follow_the_row_layout(recorder, dtype):
    nparam, K = 37, 2
    es = torch.empty(0, dtype=dtype).element_size()
    X = torch.zeros(9, 2, dtype=dtype)
    row = torch.zeros(nparam + 1 + K, dtype=dtype)
    ws = torch.zeros(64, dtype=torch.uint8)
    seed = torch.ones(K, dtype=dtype)
    prog = ops.ProgramSpec(L.PROG_RAYLEIGH).to_c()
    base = row.data_ptr()

    def sums_grad_dE(args):
        # (net, env, prog, X, n, seed, inv_n, sums, grad, energy_grad, ws, ws_bytes, stream)
        return args[7], args[8], args[9]

    ops._residual_row(L.Net(), L.Envelope(), prog, X, 9, 0.5, ws, row, nparam, seed=seed)
    kind, args = recorder.calls[-1]
    assert kind == "plain" and args[5] == seed.data_ptr() and args[6] == 0.5
    assert sums_grad_dE(args) == (base + (nparam + 1) * es, base, base + nparam * es)

    ops._residual_row(L.Net(), L.Envelope(), prog, X, 9, 0.5, ws, row, nparam, want_grad=False)
    assert sums_grad_dE(recorder.calls[-1][1]) == (base + (nparam + 1) * es, None, None)

    target = torch.zeros(K, dtype=dtype)
    ops._residual_row(L.Net(), L.Envelope(), prog, X, 9, 0.5, ws, None, nparam, sums=target, want_grad=False)
    assert sums_grad_dE(recorder.calls[-1][1]) == (target.data_ptr(), None, None)

    class Comm:              # the attributes of comm.NvlinkAllReduce that the fused exchange reads
        peers, slot, seq = L.Peers(), 128, torch.zeros(1, dtype=torch.int64)

    ops._residual_row(L.Net(), L.Envelope(), prog, X, 9, 0.5, ws, row, nparam, ar=Comm())
    kind, args = recorder.calls[-1]
    # pde_residual_loss_grad_exchange takes the row's base and derives the same offsets in C
    assert kind == "exchange" and args[7] == base and args[11] == 128 and args[12] == Comm.seq.data_ptr()


def test_row_sums_is_the_tail_of_the_row():
    row = torch.arange(10.0)
    assert torch.equal(ops._row_sums(row, 6), torch.tensor([7.0, 8.0, 9.0]))
    assert ops._row_sums(row, 6).data_ptr() == row.data_ptr() + 7 * row.element_size()


@pytest.mark.parametrize("spec", [ops.ProgramSpec(L.PROG_PINN, alpha=-0.5), ops.WanSpec(alpha=0.5, w_hi=3.0)])
def test_coefficients_fold_floats_into_the_spec(spec):
    X = torch.zeros(6, 1, dtype=torch.float64)
    out, f, beta, energy = ops._coefficients(spec, X, None, 0.75, 1.25)
    assert type(out) is type(spec) and out.beta_const == 0.75 and out.energy_const == 1.25
    assert out.alpha == spec.alpha and f is None and beta is None and energy is None
    assert spec.beta_const == 0.0 and spec.energy_const == 0.0          # the caller's spec is left as it was
    E = torch.tensor(2.0, dtype=torch.float64, requires_grad=True)
    out, _, _, energy = ops._coefficients(spec, X, None, None, E)
    assert out is spec and energy is E


def test_coefficients_pass_conforming_tensors_through_and_convert_others():
    X = torch.zeros(6, 2)
    f = torch.arange(6.0)
    _, f_out, _, _ = ops._coefficients(ops.ProgramSpec(L.PROG_MSE), X, f, None, None)
    assert f_out.data_ptr() == f.data_ptr()                             # no copy on the fast path
    beta = torch.arange(12.0, dtype=torch.float64).view(6, 2)[:, 1:]    # (6, 1), strided, other dtype
    _, _, b_out, _ = ops._coefficients(ops.ProgramSpec(L.PROG_MSE), X, None, beta, None)
    assert b_out.dtype == torch.float32 and b_out.is_contiguous() and b_out.shape == (6,)
    assert torch.equal(b_out, beta.reshape(-1).float())


def test_coefficients_refuse_a_wrong_point_count():
    X = torch.zeros(6, 1)
    for spec in (ops.ProgramSpec(L.PROG_PINN), ops.WanSpec()):
        with pytest.raises(ValueError):
            ops._coefficients(spec, X, torch.zeros(5), None, None)
        with pytest.raises(ValueError):
            ops._coefficients(spec, X, None, torch.zeros(7), None)


def test_term_weights_default_like_the_reference_and_refuse_unknown_names():
    from pde_b200 import train as T
    assert T._term_weights(None, True, False) == {'pde': 1.0, 'bc': 1e4, 'data': 0.0, 'norm': 0.0}
    assert T._term_weights({'norm': 2}, False, True, pde=3.0) == {'pde': 3.0, 'bc': 0.0, 'data': 1e3, 'norm': 2.0}
    with pytest.raises(ValueError):
        T._term_weights({'bogus': 1.0}, False, False)
