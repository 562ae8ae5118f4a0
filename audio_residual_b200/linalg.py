"""Dense linear algebra on libard_b200.so: batched fp64 symmetric eigenvalues (ard_sym_eigvals)."""
import ctypes as C

import torch

from . import lib as L


def sym_eigvals(A, overwrite=False):
    """Ascending eigenvalues [batch, D] (float64, on A's device) of the symmetric matrices A [batch, D, D] (or one [D, D]).

    A is float64 on a CUDA device; only its lower triangle is read. Every matrix of the batch goes through one call of
    ard_sym_eigvals (Householder tridiagonalisation + Sturm bisection, include/ard.h). The rows of each matrix must be contiguous;
    the matrices may sit further apart than D*D (A[b] at A + b * A.stride(0)). overwrite=True lets the solver use A as its
    scratch instead of a copy."""
    if A.dtype != torch.float64:
        raise TypeError(f"sym_eigvals: float64 matrices expected, got {A.dtype}")
    if A.device.type != "cuda":
        raise ValueError(f"sym_eigvals: matrices must be on a CUDA device, got {A.device}")
    single = A.dim() == 2
    if single:
        A = A.unsqueeze(0)
    if A.dim() != 3 or A.shape[1] != A.shape[2]:
        raise ValueError(f"sym_eigvals: [batch, D, D] expected, got {tuple(A.shape)}")
    batch, D = A.shape[0], A.shape[1]
    if batch == 0 or D == 0:
        w = torch.empty((batch, D), device=A.device, dtype=torch.float64)
        return w[0] if single else w
    rows_ok = A.stride(2) == 1 and A.stride(1) == D and (batch == 1 or A.stride(0) >= D * D)
    if not rows_ok:
        A = A.contiguous()              # a copy already
    elif not overwrite:
        A = A.clone()
    stride = A.stride(0) if batch > 1 else D * D
    lib = L.load()
    ws = lib.ard_sym_eigvals_workspace(D, batch)
    work = torch.empty(ws, device=A.device, dtype=torch.uint8)
    w = torch.empty((batch, D), device=A.device, dtype=torch.float64)
    with torch.cuda.device(A.device):
        L.check(lib.ard_sym_eigvals(C.c_void_p(A.data_ptr()), stride, D, batch, L.ptr(w), L.ptr(work), ws, L.stream_ptr()))
    return w[0] if single else w
