"""B200-native collocation-point loss step for neural-network PDE solvers.

A from-scratch CUDA (sm_100a) implementation of the hot path of
JiakangC/Neural-Network-Based-PDE-Solver: MLP forward, forward-mode derivative channels
(u, grad u, Laplacian), residual programs (PINN / Deep Ritz / WAN) and the parameter
gradient, behind the reference's own loss-function signatures.

    import pde_b200 as pb
    loss = pb.poisson.pinn_residual_loss(model, X, f, L); loss.backward()
"""
from . import _lib
from ._lib import PdeError, load as load_library
from .ops import (NO_ENVELOPE, EnvelopeSpec, ProgramSpec, WanSpec, all_reduce_grads, frozen_jets, mlp_jets,
                  residual_means, wan_means)
from . import poisson
from . import heat
from . import schrodinger
from . import train
from . import comm

__all__ = ["PdeError", "load_library", "EnvelopeSpec", "ProgramSpec", "WanSpec", "NO_ENVELOPE", "mlp_jets",
           "residual_means", "wan_means", "frozen_jets", "all_reduce_grads", "poisson", "heat", "schrodinger", "train", "comm"]
