"""Dense linear algebra on libard_b200.so: batched fp64 symmetric eigenvalues (ard_sym_eigvals) and eigenvectors (ard_sym_eigh)."""
import ctypes as C

import torch

from . import lib as L


def _solver_input(A, overwrite, name):
    """[batch, D, D] float64 CUDA matrices whose rows are contiguous, and the stride between matrices (copied unless overwrite)."""
    if A.dtype != torch.float64:
        raise TypeError(f"{name}: float64 matrices expected, got {A.dtype}")
    if A.device.type != "cuda":
        raise ValueError(f"{name}: matrices must be on a CUDA device, got {A.device}")
    single = A.dim() == 2
    if single:
        A = A.unsqueeze(0)
    if A.dim() != 3 or A.shape[1] != A.shape[2]:
        raise ValueError(f"{name}: [batch, D, D] expected, got {tuple(A.shape)}")
    batch, D = A.shape[0], A.shape[1]
    if batch and D:
        rows_ok = A.stride(2) == 1 and A.stride(1) == D and (batch == 1 or A.stride(0) >= D * D)
        if not rows_ok:
            A = A.contiguous()          # a copy already
        elif not overwrite:
            A = A.clone()
    stride = A.stride(0) if batch > 1 else D * D
    return A, stride, single


def sym_eigvals(A, overwrite=False):
    """Ascending eigenvalues [batch, D] (float64, on A's device) of the symmetric matrices A [batch, D, D] (or one [D, D]).

    A is float64 on a CUDA device; only its lower triangle is read. Every matrix of the batch goes through one call of
    ard_sym_eigvals (Householder tridiagonalisation + Sturm bisection, include/ard.h). The rows of each matrix must be contiguous;
    the matrices may sit further apart than D*D (A[b] at A + b * A.stride(0)). overwrite=True lets the solver use A as its
    scratch instead of a copy."""
    A, stride, single = _solver_input(A, overwrite, "sym_eigvals")
    batch, D = A.shape[0], A.shape[1]
    if batch == 0 or D == 0:
        w = torch.empty((batch, D), device=A.device, dtype=torch.float64)
        return w[0] if single else w
    lib = L.load()
    ws = lib.ard_sym_eigvals_workspace(D, batch)
    work = torch.empty(ws, device=A.device, dtype=torch.uint8)
    w = torch.empty((batch, D), device=A.device, dtype=torch.float64)
    with torch.cuda.device(A.device):
        L.check(lib.ard_sym_eigvals(C.c_void_p(A.data_ptr()), stride, D, batch, L.ptr(w), L.ptr(work), ws, L.stream_ptr()))
    return w[0] if single else w


def sym_eigh(A, overwrite=False):
    """(w, Q) like torch.linalg.eigh: ascending eigenvalues [batch, D] and the unit eigenvectors as the columns of Q [batch, D, D]
    (float64, on A's device) of the symmetric matrices A [batch, D, D] (or one [D, D]). Q is the .mT view of the row-major Z of
    ard_sym_eigh, so Q[b].mT[m] (row m of Z) is the eigenvector of w[b, m], contiguous. w is bitwise what sym_eigvals returns for
    the same A. Same input rules as sym_eigvals (only the lower triangle is read; overwrite=True lets the solver use A as scratch).
    Raises torch.linalg.LinAlgError when the QL iteration of some matrix did not converge: reading the per-matrix status is the
    one host synchronisation. The workspace holds one more D x D float64 matrix per batch entry (128 MB at D = 4096)."""
    A, stride, single = _solver_input(A, overwrite, "sym_eigh")
    batch, D = A.shape[0], A.shape[1]
    Z = torch.empty((batch, D, D), device=A.device, dtype=torch.float64)
    w = torch.empty((batch, D), device=A.device, dtype=torch.float64)
    if batch and D:
        lib = L.load()
        ws = lib.ard_sym_eigh_workspace(D, batch)
        work = torch.empty(ws, device=A.device, dtype=torch.uint8)
        info = torch.empty(batch, device=A.device, dtype=torch.int32)
        with torch.cuda.device(A.device):
            L.check(lib.ard_sym_eigh(C.c_void_p(A.data_ptr()), stride, D, batch, L.ptr(w), L.ptr(Z), D * D, L.ptr(info), L.ptr(work), ws,
                                     L.stream_ptr()))
        bad = torch.nonzero(info).flatten().tolist()
        if bad:
            raise torch.linalg.LinAlgError(f"sym_eigh: the QL iteration did not converge for matrices {bad} "
                                           f"({info[bad].tolist()} off-diagonals left)")
    Q = Z.mT
    return (w[0], Q[0]) if single else (w, Q)


# Workloads on which one ard_sym_eigh call is faster than torch.linalg.eigh per matrix: (largest D, smallest batch) pairs, from
# profiles/eigh_bench.json (B200, 1000 W). None of the measured ones is: 28 x 4096^2 took 16.7 s against 2.4 s, 32 x 2000^2 2.5 s
# against 0.88 s, 32 x 1152^2 0.83 s against 0.46 s, and a single matrix of 96 .. 4096 was 2.3x .. 89x slower (7.7 s against
# 0.086 s at 4096). The bound is the QL rotation generator: one thread per matrix, about 800 cycles per rotation. So every caller
# (residual.pca_on_device, analyze_attention's head components) takes torch.linalg.eigh on the device until an entry is measured.
_EIGH_LIB_MIN_BATCH = ()


def eigh_library_wins(batch, D):
    """True where one sym_eigh call of `batch` D x D matrices was measured faster than torch.linalg.eigh on each (_EIGH_LIB_MIN_BATCH)."""
    return any(D <= d and batch >= b for d, b in _EIGH_LIB_MIN_BATCH)


def eigh_batch(A):
    """(w, Q) of the float64 CUDA matrices A [batch, D, D], which it may overwrite: one sym_eigh call where that was measured
    faster (eigh_library_wins), else torch.linalg.eigh per matrix. Ascending w, eigenvectors as the columns of Q."""
    if eigh_library_wins(A.shape[0], A.shape[-1]):
        return sym_eigh(A, overwrite=True)
    outs = [torch.linalg.eigh(m) for m in A]
    return torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs])


def sign_fix(comps):
    """Rows [..., k, D] with the largest-|entry| of each row made positive (the first one on a tie): sklearn's
    svd_flip(u_based_decision=False), as residual.pca_from_moments applies it. A zero row keeps its sign."""
    idx = comps.abs().argmax(-1, keepdim=True)
    signs = torch.sign(torch.gather(comps, -1, idx))
    return comps * torch.where(signs == 0, torch.ones_like(signs), signs)
