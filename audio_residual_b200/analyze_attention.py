"""Mirror of the reference's src/analyze_attention.py on top of libard_b200.so.

extract_attention :133-157, run_PCA :13-59, save_pca_results_on_file :62-99, load_pca_csv_results :102-130.

run_PCA in the reference moves every 64x64 attention map to the host, flattens them in a triple Python loop and feeds
60 sklearn IncrementalPCA objects (~190 s per 32 clips). Here the maps stay on the GPU and each (layer, head) keeps the
sufficient statistics {n, sum x, sum x x^T} of its 4096-d samples (ard_stats_accumulate, float64 accumulators); the
spectrum is one eigendecomposition at the end. The reference's IncrementalPCA is *truncated* there (n_components =
samples of the first batch < 4096), which makes its output batch-order dependent; the exact-covariance spectrum is what
it approximates (SURVEY.md §0.3), truncated to the same number of components for schema compatibility.
"""
import csv
import os
from collections import defaultdict

import numpy as np
import torch

from .clap import batch_features
from .linalg import eigh_batch, eigh_library_wins, sign_fix, sym_eigvals
from .residual import MomentAccumulator, quantize_tensor, pad_or_truncate  # noqa: F401  (re-exported like the reference)


def _spectrum(n, s1, s2):
    """Descending eigenvalues (float64, on the GPU) of the ddof=1 covariance behind the moments {n, s1, s2}."""
    mean = s1 / n
    cov = (s2 - n * torch.outer(mean, mean)) / (n - 1)
    cov = 0.5 * (cov + cov.t())
    return torch.linalg.eigvalsh(cov).flip(0).clamp_min(0)


def _gram_spectrum(rows, n_total, D):
    """Descending ddof=1 covariance spectrum (length D, zero-padded) of the samples `rows` [n, D] with n < D, from the n x n Gram
    matrix of the centred rows (float64): same non-zero eigenvalues as the D x D covariance at (n / D)^3 of the eigen-solve."""
    X = rows.double()
    Xc = X - X.mean(0, keepdim=True)
    w = torch.linalg.eigvalsh(Xc @ Xc.t() / (n_total - 1)).flip(0).clamp_min(0)
    out = torch.zeros(D, device=rows.device, dtype=torch.float64)
    out[:w.numel()] = w[:D]
    return out


def _desc(w, Q):
    """Ascending (w, Q with eigenvectors as columns) -> descending clamped spectrum and eigenvector rows."""
    return w.flip(-1).clamp_min(0), Q.mT.flip(-2)


def _gram_components(Xc, U, D):
    """Principal axes [D, D] (rows, descending variance) of the centred rows Xc [n, D], n < D, from the Gram eigenvectors U [n, n]
    (rows, descending): the orthonormalised columns of Xc^T U^T, completed to an orthonormal basis of R^D by the complete QR."""
    Q, _ = torch.linalg.qr(Xc.mT @ U.mT, mode="complete")
    return Q.mT


def _components(n, s1, s2):
    """_spectrum with the principal axes: (descending spectrum, eigenvector rows [D, D]) of the ddof=1 covariance."""
    mean = s1 / n
    cov = (s2 - n * torch.outer(mean, mean)) / (n - 1)
    cov = 0.5 * (cov + cov.t())
    return _desc(*torch.linalg.eigh(cov))


def _gram_route_components(rows, n_total, D):
    """_gram_spectrum with the principal axes: (descending spectrum of length D, axes [D, D])."""
    X = rows.double()
    Xc = X - X.mean(0, keepdim=True)
    w, U = _desc(*torch.linalg.eigh(Xc @ Xc.t() / (n_total - 1)))
    out = torch.zeros(D, device=rows.device, dtype=torch.float64)
    out[:w.numel()] = w[:D]
    return out, _gram_components(Xc, U, D)


# Smallest group (number of matrices of one size) from which one ard_sym_eigvals call beats the per-head torch.linalg.eigvalsh loop,
# per matrix size: the first winning batch of the crossover sweep in profiles/eig_bench.json (B200, 1000 W; batches 1, 2, 4, 8, 16).
# The library pays its D column steps once per call, so a lone matrix is slower there (4096^2: 0.33 s against 0.08 s) while a batch
# shares them (28 x 4096^2: 1.0 s against 2.2 s). A size between two measured ones takes the larger one's entry.
_LIB_MIN_BATCH = ((64, 8), (256, 4), (1152, 4), (2000, 8), (4096, 8))


def _library_wins(batch, D):
    need = next((b for d, b in _LIB_MIN_BATCH if D <= d), _LIB_MIN_BATCH[-1][1])
    return batch >= need


def _solve_owned_batched(owned, accs, spectra, D, comps=None):
    """The owned heads' spectra into `spectra` rows, grouped by route and size: the D x D covariances form one group, the Gram
    matrices one group per sample count. A group at or above the measured crossover (_LIB_MIN_BATCH) is solved by one
    ard_sym_eigvals call on matrices assembled exactly as _spectrum / _gram_spectrum assemble them; a smaller group goes head by
    head through _spectrum / _gram_spectrum (also the route for CPU accumulators). A batched group holds all its matrices at once:
    28 x 128 MB = 3.8 GB for the covariance heads of one GPU at D = 4096, where the per-head route holds one.
    With `comps` (a dict) comps[i] receives head i's principal axes [D, D] (rows, descending variance, not yet sign-fixed), and
    each group, assembled the same way, goes through linalg.eigh_batch instead: one ard_sym_eigh call where that was measured
    faster than torch.linalg.eigh per head (its spectra are then bitwise those of ard_sym_eigvals), else torch.linalg.eigh per head."""
    cov = [(i, n_i) for i, n_i, r in owned if r is None]
    if cov and (eigh_library_wins(len(cov), D) if comps is not None else _library_wins(len(cov), D)):
        M = torch.empty((len(cov), D, D), device=spectra.device, dtype=torch.float64)
        for k, (i, n_i) in enumerate(cov):
            mean = accs[i].s1 / n_i
            c = (accs[i].s2 - n_i * torch.outer(mean, mean)) / (n_i - 1)
            M[k] = 0.5 * (c + c.t())
        if comps is None:
            w = sym_eigvals(M, overwrite=True).flip(-1).clamp_min(0)
        else:
            w, V = _desc(*eigh_batch(M))
            for k, (i, _) in enumerate(cov):
                comps[i] = V[k]
        spectra[[i for i, _ in cov]] = w
        del M
    else:
        for i, n_i in cov:
            if comps is None:
                spectra[i] = _spectrum(n_i, accs[i].s1, accs[i].s2)
            else:
                spectra[i], comps[i] = _components(n_i, accs[i].s1, accs[i].s2)
    grams = defaultdict(list)
    for i, n_i, r in owned:
        if r is not None:
            grams[r.shape[0]].append((i, n_i, r))
    for n, group in grams.items():
        if not (eigh_library_wins(len(group), n) if comps is not None else _library_wins(len(group), n)):
            for i, n_i, r in group:
                if comps is None:
                    spectra[i] = _gram_spectrum(r, n_i, D)
                else:
                    spectra[i], comps[i] = _gram_route_components(r, n_i, D)
            continue
        G = torch.empty((len(group), n, n), device=spectra.device, dtype=torch.float64)
        for k, (i, n_i, r) in enumerate(group):
            X = r.double()
            Xc = X - X.mean(0, keepdim=True)
            G[k] = Xc @ Xc.t() / (n_i - 1)
        if comps is None:
            w = sym_eigvals(G, overwrite=True).flip(-1).clamp_min(0)
        else:
            w, U = _desc(*eigh_batch(G))
            for k, (i, _, r) in enumerate(group):
                X = r.double()
                comps[i] = _gram_components(X - X.mean(0, keepdim=True), U[k], D)
        m = min(n, D)
        spectra[[i for i, _, _ in group], :m] = w[:, :m]


def finalize_head_spectra(accs, n_components=None, with_components=False):
    """Spectra of a list of MomentAccumulators (one per (layer, head)), as numpy arrays.
    Under torch.distributed (clip-sharded pass, SURVEY 8e) the moments are summed over ranks with the heads dealt round-robin
    to owners (`reduce` to the owner instead of an allreduce: each 4096^2 float64 matrix crosses NVLink once), every rank
    eigendecomposes only its own heads, and the spectra are exchanged in one small allreduce - the 60 serial 4096-d solves of a
    single GPU become ceil(60 / N) per GPU. After the call every accumulator's `n` is the global sample count.
    Heads that saw fewer samples than dimensions and still hold them all (MomentAccumulator.parked_rows: the last HTSAT layer
    has ONE window per clip, so a 2000-clip pass gives its 32 heads 2000 samples of 4096 dimensions) take the Gram route: the
    rows (not the D x D matrix) go to the owner and the eigen-solve is n x n (9 instead of 79 ms at n = 2000).
    On CUDA accumulators each rank solves a group of same-size heads with one ard_sym_eigvals call instead of one
    torch.linalg.eigvalsh per head, when the group is large enough for that to be faster (_solve_owned_batched); CPU accumulators
    keep _spectrum / _gram_spectrum.
    with_components=True returns (spectra, components) instead: components[i] is head i's principal axes, numpy float64
    [k, D] (k = n_components or D), rows in descending variance, sign-fixed like residual.pca_from_moments. The owner of a head
    solves it with eigenvectors (ard_sym_eigh where measured faster, spectra then bitwise as without the flag; torch.linalg.eigh
    per head otherwise, spectra within rounding, see linalg._EIGH_LIB_MIN_BATCH); Gram-route heads take the orthonormalised Xc^T U, completed to a basis of R^D. Under torch.distributed every
    rank then holds every head's components (one allreduce of a buffer that is zero outside the owner's slots): 60 heads at
    k = D = 4096 are 8 GB per rank, which is why this is opt-in."""
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    if not accs:
        return ([], []) if with_components else []
    def local_s1(a):       # first moment without disturbing parked rows (plain accumulators - the gloo tests use them - have only s1)
        if hasattr(a, "_s1"):
            return a._s1 + (a._buf[:a._fill].double().sum(0) if a._fill else 0.0)
        return a.s1

    dev, D = local_s1(accs[0]).device, accs[0].D
    rows = [a.parked_rows() if hasattr(a, "parked_rows") else None for a in accs]
    counts = torch.tensor([[float(a.n), 1.0 if r is not None else 0.0] for a, r in zip(accs, rows)], device=dev, dtype=torch.float64)
    n_loc = counts[:, 0].clone()
    if world > 1:
        # every exchange below is an allreduce (of a buffer that is zero outside this rank's slot): the collective the pass has
        # already used. A first all_gather / gather makes NCCL set up new channels, which cost seconds at 8 ranks
        both = torch.zeros((world,) + tuple(counts.shape), device=dev, dtype=torch.float64)
        both[rank] = counts
        dist.all_reduce(both)
        n_all = both[:, :, 0]                                          # [world, heads]
        n_tot = n_all.sum(0)
        parked = both[:, :, 1].min(0).values                           # every rank still holds its rows
    else:
        n_all, n_tot, parked = n_loc[None], n_loc, counts[:, 1]
    gram = [bool(parked[i] > 0) and 1 < int(n_tot[i]) < D for i in range(len(accs))]
    # global means (HeadPCA.mean_): one small allreduce of the first moments, taken before the per-head reductions below
    s1 = torch.stack([local_s1(a) for a in accs]).clone()
    if world > 1:
        dist.all_reduce(s1)
    spectra = torch.zeros((len(accs), D), device=dev, dtype=torch.float64)
    # phase 1: all the communication, head by head; phase 2: every rank eigen-solves the heads it owns. (Solving inside the first loop
    # serialises the ranks: the next head's collective waits on every GPU behind the owner's 79 ms solve - measured 5.6 s instead
    # of 1.0 s at 8 ranks.)
    owned = []
    for i, a in enumerate(accs):
        owner = i % world
        n_i = int(round(n_tot[i].item()))
        if gram[i]:
            r = rows[i]
            if world > 1:
                offs = [0]
                for k in range(world):
                    offs.append(offs[-1] + int(n_all[k, i].item()))
                allrows = torch.zeros((n_i, D), device=dev, dtype=torch.float32)
                allrows[offs[rank]:offs[rank + 1]] = r
                dist.all_reduce(allrows)                               # a few MB per head: every rank's rows in its own slot
                r = allrows
            if rank == owner:
                owned.append((i, n_i, r))
        else:
            if world > 1:
                dist.reduce(a.s1, dst=owner)
                dist.reduce(a.s2, dst=owner)
            if rank == owner:
                owned.append((i, n_i, None))
        a.n = n_i
        a.mean_global = s1[i] / max(n_i, 1)
    comps = {} if with_components else None
    if dev.type == "cuda":
        _solve_owned_batched(owned, accs, spectra, D, comps)
    else:
        for i, n_i, r in owned:
            if comps is not None:
                spectra[i], comps[i] = _gram_route_components(r, n_i, D) if r is not None else _components(n_i, accs[i].s1, accs[i].s2)
            else:
                spectra[i] = _gram_spectrum(r, n_i, D) if r is not None else _spectrum(n_i, accs[i].s1, accs[i].s2)
    if world > 1:
        dist.all_reduce(spectra)
    out = spectra.cpu().numpy()
    k = n_components or D
    spec = [out[i, :k] for i in range(len(accs))]
    if comps is None:
        return spec
    allc = torch.zeros((len(accs), k, D), device=dev, dtype=torch.float64)
    for i, c in comps.items():
        allc[i] = sign_fix(c[:k])
    if world > 1:
        dist.all_reduce(allc)
    allc = allc.cpu().numpy()
    return spec, [allc[i] for i in range(len(accs))]


class HeadPCA:
    """Stands in for a fitted sklearn IncrementalPCA: exposes the attributes the reference reads."""

    def __init__(self, D, device):
        self.acc = MomentAccumulator(D, device)
        self.first_batch = None

    def partial_fit(self, X):
        if self.first_batch is None:
            self.first_batch = X.shape[0]
        self.acc.update(X)
        return self

    def _set(self, w, n_components=None, components=None):
        """w: full descending spectrum (numpy). n_components defaults to what IncrementalPCA(n_components=None) settles on at
        its first partial_fit: min(samples of the first batch, features) (sklearn _incremental_pca.py). components: the
        principal axes (numpy rows, descending variance, at least k of them), kept as components_ when given."""
        k = n_components or min(self.first_batch or len(w), len(w))
        if components is not None:
            self.components_ = components[:k]
        mean = getattr(self.acc, "mean_global", None)
        self.mean_ = (mean if mean is not None else self.acc.s1 / self.acc.n).cpu().numpy()
        self.explained_variance_ = w[:k]
        self.explained_variance_ratio_ = w[:k] / w.sum()
        self.n_components_ = k
        self.n_samples_seen_ = self.acc.n
        return self

    def finalize(self, n_components=None, with_components=False):
        """with_components=True also sets components_ [n_components_, D] and enables transform()."""
        if not with_components:
            return self._set(finalize_head_spectra([self.acc])[0], n_components)
        spectra, comps = finalize_head_spectra([self.acc], with_components=True)
        return self._set(spectra[0], n_components, comps[0])

    def transform(self, X):
        """(X - mean_) @ components_.T: sklearn IncrementalPCA.transform with whiten=False (numpy float64)."""
        if not hasattr(self, "components_"):
            raise AttributeError("HeadPCA.transform needs components_: finalize (or run_PCA) with with_components=True")
        if isinstance(X, torch.Tensor):
            X = X.detach().cpu().numpy()
        return (np.asarray(X, dtype=np.float64) - self.mean_) @ self.components_.T


def extract_attention(clap, X, max_len=480000, data_filling="repeatpad", pad_or_truncate=False):
    """src/analyze_attention.py:133-157: block-mean attention weights per layer, list of 4 x [B*nW_l, nH_l, 64, 64]."""
    wave = batch_features(X.squeeze(1), max_len, data_filling, device=clap.device, do_pad_or_truncate=pad_or_truncate)
    enc = clap.model.audio_branch
    with torch.no_grad():
        if enc.enable_fusion:
            out = enc.encode(mel_fusion=clap.fusion_mel(wave, quantize=True), want_dict=True)
        else:
            out = enc.encode(waveform=wave, quantize=True, want_dict=True)
    return out["layers_attention"]


def run_PCA(clap, dataloader, num_layers, num_heads, components=None, data_filling="repeatpad", pad_or_truncate=False,
            with_components=False):
    """src/analyze_attention.py:13-59. Returns {layer: {head: fitted HeadPCA}}. with_components=True also gives every HeadPCA its
    components_ and transform() (finalize_head_spectra: up to 8 GB of float64 axes on every rank for 60 heads)."""
    pca_models = defaultdict(dict)
    dev = clap.device
    for l in range(num_layers):
        for h in range(num_heads[l]):
            pca_models[l][h] = HeadPCA(4096, dev)
    for batch in dataloader:
        attn = extract_attention(clap, batch[0], data_filling=data_filling, pad_or_truncate=pad_or_truncate)
        for l, layer_attn in enumerate(attn):                      # [B*nW, nH, 64, 64]
            for h in range(layer_attn.shape[1]):
                pca_models[l][h].partial_fit(layer_attn[:, h].reshape(layer_attn.shape[0], 4096))
    models = [pca_models[l][h] for l in pca_models for h in pca_models[l]]
    accs = [m.acc for m in models]
    if with_components:
        spectra, comps = finalize_head_spectra(accs, with_components=True)   # heads sharded over ranks when distributed
        for m, w, c in zip(models, spectra, comps):
            m._set(w, components, c)
    else:
        for m, w in zip(models, finalize_head_spectra(accs)):
            m._set(w, components)
    return pca_models


def save_pca_results_on_file(save_dir, dataset_name, fold, pca_models):
    """src/analyze_attention.py:62-99 (same CSV schema)."""
    os.makedirs(save_dir, exist_ok=True)
    csv_path = os.path.join(save_dir, f"{dataset_name}-fold{fold}.csv")
    with open(csv_path, mode="w", newline="") as file:
        writer = csv.writer(file)
        writer.writerow(["layer", "head", "component_index", "explained_variance", "explained_variance_ratio",
                         "participation_ratio", "intrinsic_dim"])
        for layer_idx, layer in pca_models.items():
            for head_idx, pca in layer.items():
                if not hasattr(pca, "explained_variance_"):
                    continue
                exp_var = pca.explained_variance_
                ratios = pca.explained_variance_ratio_
                cumsum = ratios.cumsum()
                intrinsic_dim = (cumsum < 0.99).sum() + 1
                pr = (exp_var.sum() ** 2) / np.sum(exp_var ** 2)
                for i, (ev, ratio) in enumerate(zip(exp_var, ratios)):
                    writer.writerow([layer_idx, head_idx, i, ev, ratio, pr if i == 0 else "", intrinsic_dim if i == 0 else ""])
    return csv_path


def load_pca_csv_results(path):
    """src/analyze_attention.py:102-130."""
    results = defaultdict(lambda: {"explained_variance": [], "explained_variance_ratio": [], "participation_ratio": None,
                                   "intrinsic_dim": None})
    with open(path, "r", newline="") as file:
        reader = csv.DictReader(file)
        for row in reader:
            key = (int(row["layer"]), int(row["head"]))
            results[key]["explained_variance"].append(float(row["explained_variance"]))
            results[key]["explained_variance_ratio"].append(float(row["explained_variance_ratio"]))
            pr = row.get("participation_ratio", "")
            if pr and results[key]["participation_ratio"] is None:
                results[key]["participation_ratio"] = float(pr)
            dim = row.get("intrinsic_dim", "")
            if dim and results[key]["intrinsic_dim"] is None:
                results[key]["intrinsic_dim"] = float(dim)
    return results
