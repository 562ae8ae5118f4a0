"""-m gpu: ard_sym_eigvals (batched fp64 symmetric eigenvalues: Householder tridiagonalisation + Sturm bisection) against
float64 LAPACK, and finalize_head_spectra / the PCA CSV on top of it against the per-head torch.linalg.eigvalsh route.

Op-level requirement: max_i |w_i - ref_i| <= 1e-11 * max_i |ref_i| per matrix. The reference is numpy.linalg.eigvalsh (float64)
for D <= 2000 and float64 torch.linalg.eigvalsh on the device at D = 4096.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from audio_residual_b200 import lib as L
from audio_residual_b200.linalg import sym_eigvals

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SIZES = [1, 2, 3, 17, 64, 255, 1152, 2000, 4096]
KINDS = ["dense", "pca", "softmax", "identity", "clustered", "diagonal", "tridiagonal", "zero", "scaled_1e-20", "scaled_1e+20"]


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _sym(M):
    return 0.5 * (M + M.t())


def _orthogonal(D, g):
    Q, R = torch.linalg.qr(torch.randn(D, D, generator=g, device=DEV, dtype=torch.float64))
    return Q * torch.sign(torch.diagonal(R))


def make_matrix(kind, D, seed):
    """One symmetric float64 [D, D] test matrix on the device."""
    g = _gen(seed)
    f64 = dict(device=DEV, dtype=torch.float64)
    if kind == "dense":
        return _sym(torch.randn(D, D, generator=g, **f64))
    if kind == "scaled_1e-20":
        return 1e-20 * _sym(torch.randn(D, D, generator=g, **f64))
    if kind == "scaled_1e+20":
        return 1e+20 * _sym(torch.randn(D, D, generator=g, **f64))
    if kind == "pca":          # covariance-like: decaying spectrum, the last D/8 eigenvalues exactly zero
        lam = torch.exp(-8.0 * torch.arange(D, **f64) / D)
        lam[D - D // 8:] = 0.0
        Q = _orthogonal(D, g)
        return _sym(Q @ (lam[:, None] * Q.t()))
    if kind == "softmax":      # centred covariance of softmax-row maps: each 64-wide row sums to 1 -> D / 64 null directions
        w = 64 if D % 64 == 0 else D
        n = D + 100
        maps = torch.softmax(2.0 * torch.randn(n, D // w, w, generator=g, **f64), dim=-1).reshape(n, D)
        Xc = maps - maps.mean(0, keepdim=True)
        return _sym(Xc.t() @ Xc / (n - 1))
    if kind == "identity":
        return torch.eye(D, **f64)
    if kind == "clustered":    # four clusters of exactly repeated eigenvalues
        lam = 1.0 + (torch.arange(D, **f64) * 4 // D)
        Q = _orthogonal(D, g)
        return _sym(Q @ (lam[:, None] * Q.t()))
    if kind == "diagonal":
        return torch.diag(torch.randn(D, generator=g, **f64))
    if kind == "tridiagonal":
        d, e = torch.randn(D, generator=g, **f64), torch.randn(max(D - 1, 0), generator=g, **f64)
        return torch.diag(d) + torch.diag(e, 1) + torch.diag(e, -1)
    if kind == "zero":
        return torch.zeros(D, D, **f64)
    raise ValueError(kind)


def reference(M):
    if M.shape[0] <= 2000:
        return torch.from_numpy(np.linalg.eigvalsh(M.cpu().numpy()))
    return torch.linalg.eigvalsh(M).cpu()


def assert_close(w, ref, what):
    w = w.cpu()
    scale = ref.abs().max().item()
    err = (w - ref).abs().max().item()
    assert err <= 1e-11 * scale, (what, err, scale, err / max(scale, 1e-300))


@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("D", SIZES)
def test_sym_eigvals(D, kind, batch):
    mats = torch.stack([make_matrix(kind, D, 1000 * D + s) for s in range(batch)])
    A = torch.tril(mats) + torch.triu(torch.full_like(mats, 123.0), 1)    # only the lower triangle is read
    w = sym_eigvals(A)
    assert w.shape == (batch, D) and w.dtype == torch.float64
    if kind == "zero":
        assert torch.count_nonzero(w).item() == 0
        return
    for b in range(batch):
        ref = reference(mats[b])
        assert torch.all(w[b, 1:] >= w[b, :-1]).item(), "ascending order"
        assert_close(w[b], ref, (kind, D, b))


def test_sym_eigvals_batch_of_28_covariances():
    """The PCA finalize's shape: 28 covariance heads of 4096 x 4096 in one call."""
    mats = torch.stack([make_matrix("pca" if s % 2 else "softmax", 4096, 77 + s) for s in range(28)])
    w = sym_eigvals(mats)
    for b in range(28):
        assert_close(w[b], torch.linalg.eigvalsh(mats[b]).cpu(), b)


@pytest.mark.parametrize("D", [17, 255, 1152])
def test_sym_eigvals_strided_batch(D):
    """Matrices further apart than D*D (stride = D*D + 37): the gaps are neither read nor written."""
    batch, stride = 3, D * D + 37
    buf = torch.full((batch, stride), 7.0, device=DEV, dtype=torch.float64)
    mats = torch.stack([make_matrix("dense", D, 5 + s) for s in range(batch)])
    buf[:, :D * D] = mats.reshape(batch, -1)
    A = buf[:, :D * D].view(batch, D, D)
    assert A.stride(0) == stride
    w = sym_eigvals(A, overwrite=True)
    assert torch.all(buf[:, D * D:] == 7.0).item()
    for b in range(batch):
        assert_close(w[b], reference(mats[b]), b)


def test_sym_eigvals_bad_arguments_raise_value_error():
    lib = L.load()
    D, batch = 8, 2
    A = torch.zeros(batch, D, D, device=DEV, dtype=torch.float64)
    w = torch.zeros(batch, D, device=DEV, dtype=torch.float64)
    ws = lib.ard_sym_eigvals_workspace(D, batch)
    assert ws > 0
    work = torch.zeros(ws, device=DEV, dtype=torch.uint8)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    good = dict(A=p(A), stride=D * D, D=D, batch=batch, w=p(w), work=p(work), work_bytes=ws)
    bad = [dict(D=0), dict(D=-3), dict(batch=0), dict(stride=D * D - 1), dict(A=None), dict(w=None), dict(work=None),
           dict(work_bytes=ws - 1)]
    for change in bad:
        a = {**good, **change}
        rc = lib.ard_sym_eigvals(a["A"], a["stride"], a["D"], a["batch"], a["w"], a["work"], a["work_bytes"], L.stream_ptr())
        assert rc == L.ARD_ERR_SHAPE, change
        with pytest.raises(ValueError):
            L.check(rc)
    torch.cuda.synchronize()
    assert torch.count_nonzero(w).item() == 0          # nothing ran
    # the Python op: dtype and device are checked before the call
    with pytest.raises(TypeError):
        sym_eigvals(A.float())
    with pytest.raises(ValueError):
        sym_eigvals(A.cpu())
    with pytest.raises(ValueError):
        sym_eigvals(torch.zeros(2, 3, 4, device=DEV, dtype=torch.float64))


# ------------------------------------------------------------------------------------------------ end to end: run_PCA finalize
def test_finalize_head_spectra_matches_per_head_eigvalsh(tmp_path):
    """A real run_PCA pass on HTSAT-tiny (4 clips: every head keeps its rows, so all 60 take the Gram route), then again with the
    rows of layers 0-2 folded into their moments (28 heads on the 4096 x 4096 covariance route, 32 on the Gram route, in one call).
    Both against _spectrum / _gram_spectrum on the same moments / rows, to 1e-10 of the top eigenvalue; n_components truncation;
    the CSV's participation ratio (1e-9 relative) and intrinsic dimension (equal)."""
    import gpu_checks as G
    from audio_residual_b200 import analyze_attention as A
    from audio_residual_b200 import weights as W

    clap, _, _ = G.make_encoder("tiny")
    g = torch.Generator().manual_seed(5)
    batches = [(W.make_clips(2, seed=41).unsqueeze(1), torch.tensor([0, 1])),
               ((0.1 * torch.randn(2, 300000, generator=g)).clamp_(-1, 1).unsqueeze(1), torch.tensor([2, 3]))]
    models = A.run_PCA(clap, batches, 4, [4, 8, 16, 32])
    heads = [models[l][h] for l in models for h in models[l]]
    accs = [m.acc for m in heads]
    D = 4096

    def reference_spectra():
        out = []
        for a in accs:
            r = a.parked_rows()
            out.append((A._gram_spectrum(r, a.n, D) if r is not None else A._spectrum(a.n, a.s1, a.s2)).cpu().numpy())
        return out

    def check(spectra, ref):
        for i, (w, rw) in enumerate(zip(spectra, ref)):
            assert w.shape == (D,)
            err = np.abs(w - rw).max()
            assert err <= 1e-10 * rw[0], (i, err, rw[0])

    assert all(a.parked_rows() is not None for a in accs)
    ref = reference_spectra()
    spectra = A.finalize_head_spectra(accs)
    check(spectra, ref)
    trunc = A.finalize_head_spectra(accs, n_components=64)
    assert all(t.shape == (64,) and np.array_equal(t, s[:64]) for t, s in zip(trunc, spectra))

    # CSV summaries from the solver's spectra vs from the reference spectra
    for m, w in zip(heads, spectra):
        m._set(w)
    back = A.load_pca_csv_results(A.save_pca_results_on_file(str(tmp_path), "synthetic", 0, models))
    for (l, h), rw in zip([(l, h) for l in models for h in models[l]], ref):
        k = models[l][h].n_components_
        ev, ratio = rw[:k], rw[:k] / rw.sum()
        pr = ev.sum() ** 2 / np.sum(ev ** 2)
        idim = (ratio.cumsum() < 0.99).sum() + 1
        assert abs(back[(l, h)]["participation_ratio"] - pr) <= 1e-9 * pr, (l, h)
        assert back[(l, h)]["intrinsic_dim"] == idim, (l, h)

    # covariance route for layers 0-2 (reading s2 folds the parked rows into the moments), Gram route for layer 3
    for l in (0, 1, 2):
        for h in models[l]:
            models[l][h].acc.s2
    assert sum(a.parked_rows() is None for a in accs) == 28
    ref = reference_spectra()
    check(A.finalize_head_spectra(accs), ref)


def test_finalize_routes_small_groups_per_head_and_large_groups_to_the_library():
    """Below the measured crossover (one 4096-d covariance head, HeadPCA.finalize) the per-head _spectrum route runs, bit for bit;
    at it (8 heads) one ard_sym_eigvals call does, to 1e-10 of the top eigenvalue."""
    from audio_residual_b200 import analyze_attention as A
    from audio_residual_b200.residual import MomentAccumulator

    g = torch.Generator(device=DEV).manual_seed(3)
    accs = []
    for h in range(8):
        a = MomentAccumulator(4096, DEV, min_rows=0)
        a.update(torch.softmax(2.0 * torch.randn(2100, 64, 64, generator=g, device=DEV), dim=-1).reshape(2100, 4096))
        accs.append(a)
    assert not A._library_wins(1, 4096) and A._library_wins(8, 4096)
    ref = [A._spectrum(a.n, a.s1, a.s2).cpu().numpy() for a in accs]
    one = A.finalize_head_spectra(accs[:1])[0]
    assert np.array_equal(one, ref[0])
    calls = []
    real = A.sym_eigvals
    A.sym_eigvals = lambda M, **kw: calls.append(M.shape) or real(M, **kw)
    try:
        got = A.finalize_head_spectra(accs)
    finally:
        A.sym_eigvals = real
    assert calls == [(8, 4096, 4096)]
    for w, rw in zip(got, ref):
        assert np.abs(w - rw).max() <= 1e-10 * rw[0]
