"""ctypes binding of libpde_b200.so (include/pde_b200.h).

The library is the product; there is no Python or CPU fallback.  ``load()`` raises if the
shared object has not been built (``python __graft_entry__.py build`` or ``make -C csrc``).
"""
from __future__ import annotations

import ctypes as C
import os

MAX_LINEAR, MAX_DIM, MAX_NODES, MAX_Q = 8, 5, 8, 4
F32, F64 = 0, 1
ACT_SIN, ACT_TANH = 0, 1
ENV_NONE, ENV_POLY, ENV_EXPWIN = 0, 1, 2
PROG_PINN, PROG_DRM, PROG_RAYLEIGH, PROG_MSE, PROG_FLUX = 1, 2, 3, 4, 5

EXPORTS = [
    "pde_abi_version", "pde_strerror", "pde_param_count", "pde_jet_channels", "pde_program_quantities",
    "pde_program_order", "pde_workspace_bytes", "pde_jets_forward", "pde_jets_backward",
    "pde_residual_loss_grad", "pde_wan_pointwise", "pde_query_path", "pde_sample_points_rhs", "pde_adam_step",
    "pde_keep_best", "pde_peer_bytes", "pde_peer_alloc", "pde_peer_open", "pde_peer_close", "pde_peer_free",
    "pde_allreduce_oneshot", "pde_query_jets_path", "pde_set_kernel_path", "pde_kernel_path", "pde_last_kernel_path",
    "pde_launch_count", "pde_set_exchange_timeout", "pde_exchange_errors", "pde_residual_loss_grad_exchange", "pde_wan_scalars",
    "pde_sample_faces_rhs",
]
MAX_PEERS = 8


class Net(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("dim", C.c_int32), ("n_linear", C.c_int32), ("activation", C.c_int32),
                ("widths", C.c_int32 * (MAX_LINEAR + 1)), ("W", C.c_void_p * MAX_LINEAR), ("b", C.c_void_p * MAX_LINEAR)]


class Envelope(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_nodes", C.c_int32 * MAX_DIM), ("lo", C.c_double), ("hi", C.c_double),
                ("nodes", (C.c_double * MAX_NODES) * MAX_DIM)]


class Program(C.Structure):
    _fields_ = [("kind", C.c_int32), ("faces", C.c_int32), ("alpha", C.c_double), ("beta_const", C.c_double),
                ("energy_const", C.c_double), ("f", C.c_void_p), ("beta", C.c_void_p), ("energy", C.c_void_p)]


class Wan(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("dim", C.c_int32), ("alpha", C.c_double), ("beta_const", C.c_double),
                ("energy_const", C.c_double), ("w_lo", C.c_double), ("w_hi", C.c_double), ("eps_den", C.c_double),
                ("f", C.c_void_p), ("beta", C.c_void_p), ("energy", C.c_void_p),
                ("env_u", Envelope), ("env_v", Envelope)]


class Adam(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("n_tensors", C.c_int32), ("lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double), ("grad_scale", C.c_double),
                ("param", C.c_void_p * (2 * MAX_LINEAR + 1)), ("numel", C.c_int64 * (2 * MAX_LINEAR + 1))]


class Peers(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("base", C.c_void_p * MAX_PEERS)]


class PdeError(RuntimeError):
    pass


_LIB = None


def lib_path():
    if os.environ.get("PDE_B200_LIB"):   # development: an alternative build of the same library
        return os.environ["PDE_B200_LIB"]
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libpde_b200.so")


def load():
    """Load the CUDA library; fail loudly when it is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise PdeError(f"{path} not built: run `python __graft_entry__.py build` (nvcc, sm_100a). "
                       "There is no CPU fallback for the collocation kernels.")
    lib = C.CDLL(path)
    vp, sz, i32, i64, dbl = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64, C.c_double
    lib.pde_abi_version.restype = C.c_int
    lib.pde_strerror.restype = C.c_char_p
    lib.pde_strerror.argtypes = [C.c_int]
    lib.pde_param_count.argtypes = [C.POINTER(Net), C.POINTER(i64)]
    lib.pde_jet_channels.argtypes = [i32, i32]
    lib.pde_program_quantities.argtypes = [i32]
    lib.pde_program_order.argtypes = [i32]
    lib.pde_workspace_bytes.argtypes = [C.POINTER(Net), i32, i64, C.POINTER(sz)]
    lib.pde_jets_forward.argtypes = [C.POINTER(Net), i32, vp, i64, vp, vp, sz, vp]
    lib.pde_jets_backward.argtypes = [C.POINTER(Net), i32, vp, i64, vp, vp, vp, sz, vp]
    lib.pde_residual_loss_grad.argtypes = [C.POINTER(Net), C.POINTER(Envelope), C.POINTER(Program), vp, i64, vp, dbl,
                                           vp, vp, vp, vp, sz, vp]
    lib.pde_residual_loss_grad_exchange.argtypes = [C.POINTER(Net), C.POINTER(Envelope), C.POINTER(Program), vp, i64, vp, dbl,
                                                    vp, vp, sz, C.POINTER(Peers), i64, vp, vp]
    lib.pde_wan_scalars.argtypes = [i32, i32, vp, C.POINTER(dbl), vp, vp, vp]
    lib.pde_query_path.argtypes = [C.POINTER(Net), C.POINTER(Program), i64]
    lib.pde_wan_pointwise.argtypes = [C.POINTER(Wan), vp, i64, vp, vp, vp, dbl, vp, vp, vp, vp, sz, vp]
    lib.pde_sample_points_rhs.argtypes = [i32, i32, i64, dbl, dbl, C.c_uint64, C.c_uint64, vp, C.POINTER(dbl), dbl, vp, vp,
                                          vp, vp, vp]
    lib.pde_sample_faces_rhs.argtypes = [i32, i32, i64, i32, dbl, dbl, C.c_uint64, C.c_uint64, vp, C.POINTER(dbl), dbl, vp,
                                         vp, vp]
    lib.pde_adam_step.argtypes = [C.POINTER(Adam), vp, vp, vp, vp, vp]
    lib.pde_keep_best.argtypes = [C.POINTER(Adam), vp, vp, vp, vp, vp, vp]
    lib.pde_peer_bytes.argtypes = [i32, i64, C.POINTER(sz)]
    lib.pde_peer_alloc.argtypes = [sz, C.POINTER(vp), C.c_char_p]
    lib.pde_peer_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    lib.pde_peer_close.argtypes = [vp]
    lib.pde_peer_free.argtypes = [vp]
    lib.pde_allreduce_oneshot.argtypes = [C.POINTER(Peers), i32, vp, i64, i64, vp, vp]
    lib.pde_set_exchange_timeout.argtypes = [dbl]
    lib.pde_exchange_errors.argtypes = [C.POINTER(Peers), C.POINTER(C.c_uint32), vp]
    lib.pde_query_jets_path.argtypes = [C.POINTER(Net), i32, i64]
    lib.pde_set_kernel_path.argtypes = [i32]
    for name in EXPORTS:
        if name not in ("pde_strerror", "pde_launch_count"):
            getattr(lib, name).restype = C.c_int
    lib.pde_launch_count.restype = C.c_uint64
    if lib.pde_abi_version() != 1:
        raise PdeError("libpde_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def check(status, what=""):
    if status != 0:
        msg = load().pde_strerror(status).decode()
        if status == -2:
            raise NotImplementedError(f"{what}: {msg}")
        if status == -1:
            raise ValueError(f"{what}: {msg}")
        raise PdeError(f"{what}: {msg} (status {status})")
