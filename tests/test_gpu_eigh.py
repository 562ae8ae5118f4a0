"""-m gpu: ard_sym_eigh (batched fp64 symmetric eigenvectors: the ard_sym_eigvals reduction keeping its reflectors, implicit QL on
the tridiagonal matrix, blocked back-transformation), and the PCA components built on it (compute_pca_components, HeadPCA /
run_PCA with_components=True).

Op-level requirements per matrix: w is torch.equal to sym_eigvals on the same input; max_m ||A z_m - w_m z_m||_2 <= 1e-11 max|w|;
max|Z Z^T - I| <= 1e-11; every eigenvector whose eigenvalue is at least 1e-3 max|w| away from every other one equals float64
LAPACK's up to sign to 1e-9 (numpy.linalg.eigh, torch.linalg.eigh on the device at D = 4096); info == 0. Clustered and zero
spectra are judged by residual and orthogonality alone, which is what defines a correct basis of an invariant subspace.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from audio_residual_b200 import lib as L
from audio_residual_b200.linalg import sym_eigh, sym_eigvals
from test_gpu_eig import DEV, KINDS, make_matrix

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 3, 17, 64, 96, 192, 384, 768, 1024, 1152, 4096]


def reference_eigh(M):
    if M.shape[0] < 4096:
        w, v = np.linalg.eigh(M.cpu().numpy())
        return torch.from_numpy(w), torch.from_numpy(v)
    w, v = torch.linalg.eigh(M)
    return w.cpu(), v.cpu()


def check_eigh(M, w, Q, what):
    """M [D, D] (full symmetric), w [D], Q [D, D] with the eigenvectors as columns."""
    D = M.shape[0]
    scale = max(w.abs().max().item(), 1e-300)
    R = M @ Q - Q * w[None, :]
    res = torch.linalg.vector_norm(R, dim=0).max().item()
    assert res <= 1e-11 * scale or (scale == 1e-300 and res == 0.0), (what, "residual", res, scale)
    orth = (Q.mT @ Q - torch.eye(D, device=Q.device, dtype=torch.float64)).abs().max().item()
    assert orth <= 1e-11, (what, "orthogonality", orth)
    if scale == 1e-300:
        return
    rw, rv = reference_eigh(M)
    wc = w.cpu()
    gap = torch.full((D,), float("inf"), dtype=torch.float64)
    if D > 1:
        d = wc[1:] - wc[:-1]
        gap[1:] = torch.minimum(gap[1:], d)
        gap[:-1] = torch.minimum(gap[:-1], d)
    sep = gap >= 1e-3 * scale
    if sep.any():
        Qc = Q.cpu()[:, sep]
        Rc = rv[:, sep]
        sign = torch.sign((Qc * Rc).sum(0))
        err = (Qc - Rc * sign[None, :]).abs().max().item()
        assert err <= 1e-9, (what, "vs LAPACK", err, int(sep.sum()))


@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("D", SIZES)
def test_sym_eigh(D, kind, batch):
    if D == 4096 and batch == 3 and kind not in ("dense", "pca", "softmax"):
        pytest.skip("batch 3 at 4096 is covered by the dense / pca / softmax families and the batch of 28")
    mats = torch.stack([make_matrix(kind, D, 1000 * D + s) for s in range(batch)])
    A = torch.tril(mats) + torch.triu(torch.full_like(mats, 123.0), 1)    # only the lower triangle is read
    w, Q = sym_eigh(A)
    assert w.shape == (batch, D) and Q.shape == (batch, D, D) and w.dtype == Q.dtype == torch.float64
    assert torch.equal(w, sym_eigvals(A))
    assert torch.equal(A[:, 0, 0], torch.tril(mats)[:, 0, 0])           # overwrite=False works on a copy
    for b in range(batch):
        check_eigh(mats[b], w[b], Q[b], (kind, D, b))


def test_sym_eigh_batch_of_28_covariances():
    """The PCA finalize's shape: 28 covariance heads of 4096 x 4096 in one call."""
    mats = torch.stack([make_matrix("pca" if s % 2 else "softmax", 4096, 77 + s) for s in range(28)])
    w, Q = sym_eigh(mats)
    assert torch.equal(w, sym_eigvals(mats))
    for b in range(0, 28, 3):
        check_eigh(mats[b], w[b], Q[b], b)
    for b in range(28):                    # residual and orthogonality on every one (cheap on the device)
        M, q, wb = mats[b], Q[b], w[b]
        scale = wb.abs().max().item()
        assert torch.linalg.vector_norm(M @ q - q * wb[None, :], dim=0).max().item() <= 1e-11 * scale, b
        assert (q.mT @ q - torch.eye(4096, device=DEV, dtype=torch.float64)).abs().max().item() <= 1e-11, b


@pytest.mark.parametrize("D", [17, 384, 1152])
def test_sym_eigh_strided_batch(D):
    """Matrices further apart than D*D (stride = D*D + 37): the gaps are neither read nor written."""
    batch, stride = 3, D * D + 37
    buf = torch.full((batch, stride), 7.0, device=DEV, dtype=torch.float64)
    mats = torch.stack([make_matrix("dense", D, 5 + s) for s in range(batch)])
    buf[:, :D * D] = mats.reshape(batch, -1)
    A = buf[:, :D * D].view(batch, D, D)
    assert A.stride(0) == stride
    ref_w = sym_eigvals(A)
    w, Q = sym_eigh(A, overwrite=True)
    assert torch.all(buf[:, D * D:] == 7.0).item()
    assert torch.equal(w, ref_w)
    for b in range(batch):
        check_eigh(mats[b], w[b], Q[b], b)


def test_sym_eigh_bad_arguments_raise_value_error():
    lib = L.load()
    D, batch = 8, 2
    A = torch.zeros(batch, D, D, device=DEV, dtype=torch.float64)
    w = torch.zeros(batch, D, device=DEV, dtype=torch.float64)
    Z = torch.zeros(batch, D, D, device=DEV, dtype=torch.float64)
    info = torch.full((batch,), -1, device=DEV, dtype=torch.int32)
    ws = lib.ard_sym_eigh_workspace(D, batch)
    assert ws > lib.ard_sym_eigvals_workspace(D, batch) > 0
    assert lib.ard_sym_eigh_workspace(0, 1) == 0 and lib.ard_sym_eigh_workspace(4, 0) == 0
    work = torch.zeros(ws, device=DEV, dtype=torch.uint8)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    good = dict(A=p(A), stride=D * D, D=D, batch=batch, w=p(w), Z=p(Z), zstride=D * D, info=p(info), work=p(work), work_bytes=ws)
    bad = [dict(D=0), dict(D=-3), dict(batch=0), dict(batch=65536), dict(stride=D * D - 1), dict(A=None), dict(w=None),
           dict(work=None), dict(work_bytes=ws - 1), dict(Z=None), dict(info=None), dict(zstride=D * D - 1), dict(D=12289)]
    for change in bad:
        a = {**good, **change}
        rc = lib.ard_sym_eigh(a["A"], a["stride"], a["D"], a["batch"], a["w"], a["Z"], a["zstride"], a["info"], a["work"],
                              a["work_bytes"], L.stream_ptr())
        assert rc == L.ARD_ERR_SHAPE, change
        with pytest.raises(ValueError):
            L.check(rc)
    torch.cuda.synchronize()
    assert torch.count_nonzero(w).item() == 0 and torch.count_nonzero(Z).item() == 0   # nothing ran
    assert torch.all(info == -1).item()
    with pytest.raises(TypeError):
        sym_eigh(A.float())
    with pytest.raises(ValueError):
        sym_eigh(A.cpu())
    with pytest.raises(ValueError):
        sym_eigh(torch.zeros(2, 3, 4, device=DEV, dtype=torch.float64))


def test_sym_eigh_single_matrix_and_empty():
    M = make_matrix("dense", 50, 9)
    w, Q = sym_eigh(M)
    assert w.shape == (50,) and Q.shape == (50, 50)
    check_eigh(M, w, Q, "single")
    w0, Q0 = sym_eigh(torch.zeros(0, 5, 5, device=DEV, dtype=torch.float64))
    assert w0.shape == (0, 5) and Q0.shape == (0, 5, 5)


# ------------------------------------------------------------------------------------------------ PCA components on the device
def _separated(w, rel=1e-3):
    """Mask of the entries of a descending spectrum at least rel * max away from both neighbours."""
    w = np.asarray(w)
    gap = np.full(len(w), np.inf)
    d = np.abs(np.diff(w))
    gap[1:] = np.minimum(gap[1:], d)
    gap[:-1] = np.minimum(gap[:-1], d)
    return gap >= rel * np.abs(w).max()


def _sign_fixed_rows(v):
    """numpy eigh columns (ascending) -> rows in descending order with pca_from_moments' sign rule."""
    v = v[:, ::-1].T
    return v * np.where(np.sign(v[np.arange(len(v)), np.abs(v).argmax(1)]) == 0, 1.0,
                        np.sign(v[np.arange(len(v)), np.abs(v).argmax(1)]))[:, None]


@pytest.mark.parametrize("route", ["measured", "library"])
def test_compute_pca_components_on_device_matches_pca_from_moments(route, monkeypatch):
    """Every HTSAT-tiny layer (96 .. 768 wide), with and without n_components: the dict of the device route against
    pca_from_moments (numpy) on the same moments; on the measured route table (linalg._EIGH_LIB_MIN_BATCH) and with the solve
    forced onto one ard_sym_eigh call."""
    import gpu_checks as G
    from audio_residual_b200 import linalg as LA
    from audio_residual_b200 import residual as R
    from audio_residual_b200 import weights as W

    if route == "library":
        monkeypatch.setattr(LA, "_EIGH_LIB_MIN_BATCH", ((4096, 1),))
        calls = []
        real_eigh = LA.sym_eigh
        monkeypatch.setattr(LA, "sym_eigh", lambda A, **kw: calls.append(A.shape) or real_eigh(A, **kw))

    clap, _, _ = G.make_encoder("tiny")
    batches = [(W.make_clips(2, seed=61 + i).unsqueeze(1), torch.zeros(2, dtype=torch.long)) for i in range(2)]
    seen = []
    real = R.MomentAccumulator.pca

    def spy(self, n_components=None):
        seen.append((self.n, self.s1.cpu().numpy(), self.s2.cpu().numpy()))
        return real(self, n_components)
    R.MomentAccumulator.pca = spy
    try:
        for layer in range(4):
            for k in (None, 16):
                got = R.compute_pca_components(clap, batches, layer, n_components=k)
                n, s1, s2 = seen[-1]
                ref = R.pca_from_moments(n, s1, s2, k)
                full = R.pca_from_moments(n, s1, s2)
                assert sorted(got) == sorted(ref)
                for key in ("n_components", "input_dim", "num_samples"):
                    assert got[key] == ref[key], (layer, k, key)
                D = ref["input_dim"]
                kk = ref["n_components"]
                assert got["components"].shape == (kk, D) and got["components"].dtype == np.float64
                assert np.abs(got["mean"] - ref["mean"]).max() <= 1e-15 * np.abs(ref["mean"]).max()
                top = full["explained_variance"][0]
                assert np.abs(got["explained_variance"] - ref["explained_variance"]).max() <= 1e-10 * top, (layer, k)
                assert np.abs(got["explained_variance_ratio"] - ref["explained_variance_ratio"]).max() <= 1e-10, (layer, k)
                sep = _separated(full["explained_variance"])[:kk]
                assert sep.sum() >= 4, (layer, int(sep.sum()))
                err = np.abs(got["components"][sep] - ref["components"][sep]).max()
                assert err <= 1e-8, (layer, k, err)
                c = got["components"]
                assert np.abs(c @ c.T - np.eye(kk)).max() <= 1e-11
    finally:
        R.MomentAccumulator.pca = real
    if route == "library":
        assert len(calls) == 8 and all(c[0] == 1 for c in calls)


def test_head_pca_components_match_incremental_pca():
    """HeadPCA(64, cuda) fed in batches against sklearn IncrementalPCA(n_components=None) fed the same float64 batches on full-rank
    data. The samples are small integers, so the device moments are exact and the two agree to float64 rounding."""
    from sklearn.decomposition import IncrementalPCA

    from audio_residual_b200.analyze_attention import HeadPCA
    rng = np.random.default_rng(4)
    X = rng.integers(-8, 9, size=(600, 64)) * (1 + np.arange(64) % 5)
    X = X.astype(np.float64) + 3.0
    hp, ip = HeadPCA(64, DEV), IncrementalPCA(n_components=None)
    for b in range(6):
        xb = X[100 * b:100 * (b + 1)]
        hp.partial_fit(torch.from_numpy(xb).to(DEV))
        ip.partial_fit(xb)
    hp.finalize(with_components=True)
    assert hp.n_components_ == ip.n_components_ == 64
    assert hp.components_.shape == (64, 64) and hp.components_.dtype == np.float64
    assert np.abs(hp.explained_variance_ - ip.explained_variance_).max() <= 1e-10 * ip.explained_variance_[0]
    assert np.abs(hp.components_ - ip.components_).max() <= 1e-9
    Y = rng.standard_normal((50, 64)) * 10
    ref = ip.transform(Y)
    assert np.abs(hp.transform(Y) - ref).max() <= 1e-9 * np.abs(ref).max()
    assert np.abs(hp.transform(torch.from_numpy(Y).to(DEV)) - ref).max() <= 1e-9 * np.abs(ref).max()
    plain = HeadPCA(64, DEV)
    plain.partial_fit(torch.from_numpy(X).to(DEV))
    plain.finalize()
    assert not hasattr(plain, "components_")
    with pytest.raises(AttributeError):
        plain.transform(Y)


@pytest.mark.parametrize("route", ["measured", "library"])
def test_run_pca_with_components_both_routes(route, monkeypatch):
    """run_PCA(with_components=True) on HTSAT-tiny (4 clips: all 60 heads on the Gram route), then the 28 heads of layers 0-2 on the
    covariance route (their parked rows folded into the moments). Components against torch float64 eigh of the covariance of the
    same maps (Gram route) or of the same moments (covariance route, whose moments are fp32-grade); spectra unchanged by the flag
    (bitwise when the groups go through ard_sym_eigh, to 1e-12 of the top on the per-head torch.linalg.eigh route the measured
    table picks); no components_ without it. route="library" forces every group onto one ard_sym_eigh call."""
    import gpu_checks as G
    from audio_residual_b200 import analyze_attention as A
    from audio_residual_b200 import linalg as LA
    from audio_residual_b200 import weights as W

    if route == "library":
        monkeypatch.setattr(A, "eigh_library_wins", lambda batch, D: True)
        calls = []
        real_eigh = LA.sym_eigh
        monkeypatch.setattr(LA, "sym_eigh", lambda M, **kw: calls.append(tuple(M.shape)) or real_eigh(M, **kw))
        monkeypatch.setattr(LA, "_EIGH_LIB_MIN_BATCH", ((4096, 1),))

    def same_spectrum(a, b):
        if route == "library":
            return np.array_equal(a, b)
        return np.abs(a - b).max() <= 1e-12 * b[0]

    clap, _, _ = G.make_encoder("tiny")
    g = torch.Generator().manual_seed(5)
    batches = [(W.make_clips(2, seed=41).unsqueeze(1), torch.tensor([0, 1])),
               ((0.1 * torch.randn(2, 300000, generator=g)).clamp_(-1, 1).unsqueeze(1), torch.tensor([2, 3]))]
    plain = A.run_PCA(clap, batches, 4, [4, 8, 16, 32])
    assert not any(hasattr(plain[l][h], "components_") for l in plain for h in plain[l])
    models = A.run_PCA(clap, batches, 4, [4, 8, 16, 32], with_components=True)
    heads = [models[l][h] for l in models for h in models[l]]
    pheads = [plain[l][h] for l in plain for h in plain[l]]
    accs = [m.acc for m in heads]
    assert all(a.parked_rows() is not None for a in accs)
    for m, p in zip(heads, pheads):
        assert same_spectrum(m.explained_variance_, p.explained_variance_)
        assert m.components_.shape == (m.n_components_, 4096)

    def check(i, comps, cov, spec):
        w, v = torch.linalg.eigh(cov)
        w = w.flip(0).clamp_min(0).cpu().numpy()
        ref = _sign_fixed_rows(v.cpu().numpy())
        k = comps.shape[0]
        sep = _separated(w)[:k] & (w[:k] > 1e-6 * w[0])
        assert sep.sum() >= 1, i
        assert np.abs(spec - w[:len(spec)]).max() <= 1e-10 * w[0], i
        assert np.abs(comps[sep] - ref[:k][sep]).max() <= 1e-8, (i, np.abs(comps[sep] - ref[:k][sep]).max())
        assert np.abs(comps @ comps.T - np.eye(k)).max() <= 1e-10, i

    rows = [a.parked_rows().double().clone() for a in accs]
    for i in (0, 5, 20, 40, 59):                                       # Gram route (the HeadPCA's truncated components_)
        X = rows[i]
        check(i, heads[i].components_, torch.cov(X.t(), correction=1), heads[i].explained_variance_)
    for l in (0, 1, 2):                                                # covariance route for the 28 heads of layers 0-2
        for h in models[l]:
            models[l][h].acc.s2
    spectra_c, comps_c = A.finalize_head_spectra(accs, with_components=True)
    spectra_p = A.finalize_head_spectra(accs)
    for i in range(60):
        assert same_spectrum(spectra_c[i], spectra_p[i]), i
        assert comps_c[i].shape == (4096, 4096)
    if route == "library":
        assert (28, 4096, 4096) in calls and len(calls) > 1          # the covariance group and the Gram groups
    for i in (0, 13, 27, 30):
        a = accs[i]
        if i < 28:
            mean = a.s1 / a.n
            cov = (a.s2 - a.n * torch.outer(mean, mean)) / (a.n - 1)
            cov = 0.5 * (cov + cov.t())
            maps = torch.cov(rows[i].t(), correction=1)
            w_maps = torch.linalg.eigvalsh(maps).flip(0).cpu().numpy()
            assert np.abs(spectra_c[i][:32] - w_maps[:32]).max() <= 1e-4 * w_maps[0], i   # fp32-grade moments vs the maps
        else:
            cov = torch.cov(rows[i].t(), correction=1)
        check(i, comps_c[i], cov, spectra_c[i])
