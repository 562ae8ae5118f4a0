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
from .linalg import sym_eigvals
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


# Smallest group (number of matrices of one size) from which one ard_sym_eigvals call beats the per-head torch.linalg.eigvalsh loop,
# per matrix size: the first winning batch of the crossover sweep in profiles/eig_bench.json (B200, 1000 W; batches 1, 2, 4, 8, 16).
# The library pays its D column steps once per call, so a lone matrix is slower there (4096^2: 0.33 s against 0.08 s) while a batch
# shares them (28 x 4096^2: 1.0 s against 2.2 s). A size between two measured ones takes the larger one's entry.
_LIB_MIN_BATCH = ((64, 8), (256, 4), (1152, 4), (2000, 8), (4096, 8))


def _library_wins(batch, D):
    need = next((b for d, b in _LIB_MIN_BATCH if D <= d), _LIB_MIN_BATCH[-1][1])
    return batch >= need


def _solve_owned_batched(owned, accs, spectra, D):
    """The owned heads' spectra into `spectra` rows, grouped by route and size: the D x D covariances form one group, the Gram
    matrices one group per sample count. A group at or above the measured crossover (_LIB_MIN_BATCH) is solved by one
    ard_sym_eigvals call on matrices assembled exactly as _spectrum / _gram_spectrum assemble them; a smaller group goes head by
    head through _spectrum / _gram_spectrum (also the route for CPU accumulators). A batched group holds all its matrices at once:
    28 x 128 MB = 3.8 GB for the covariance heads of one GPU at D = 4096, where the per-head route holds one."""
    cov = [(i, n_i) for i, n_i, r in owned if r is None]
    if cov and _library_wins(len(cov), D):
        M = torch.empty((len(cov), D, D), device=spectra.device, dtype=torch.float64)
        for k, (i, n_i) in enumerate(cov):
            mean = accs[i].s1 / n_i
            c = (accs[i].s2 - n_i * torch.outer(mean, mean)) / (n_i - 1)
            M[k] = 0.5 * (c + c.t())
        w = sym_eigvals(M, overwrite=True).flip(-1).clamp_min(0)
        spectra[[i for i, _ in cov]] = w
        del M
    else:
        for i, n_i in cov:
            spectra[i] = _spectrum(n_i, accs[i].s1, accs[i].s2)
    grams = defaultdict(list)
    for i, n_i, r in owned:
        if r is not None:
            grams[r.shape[0]].append((i, n_i, r))
    for n, group in grams.items():
        if not _library_wins(len(group), n):
            for i, n_i, r in group:
                spectra[i] = _gram_spectrum(r, n_i, D)
            continue
        G = torch.empty((len(group), n, n), device=spectra.device, dtype=torch.float64)
        for k, (i, n_i, r) in enumerate(group):
            X = r.double()
            Xc = X - X.mean(0, keepdim=True)
            G[k] = Xc @ Xc.t() / (n_i - 1)
        w = sym_eigvals(G, overwrite=True).flip(-1).clamp_min(0)
        m = min(n, D)
        spectra[[i for i, _, _ in group], :m] = w[:, :m]


def finalize_head_spectra(accs, n_components=None):
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
    keep _spectrum / _gram_spectrum."""
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    if not accs:
        return []
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
    if dev.type == "cuda":
        _solve_owned_batched(owned, accs, spectra, D)
    else:
        for i, n_i, r in owned:
            spectra[i] = _gram_spectrum(r, n_i, D) if r is not None else _spectrum(n_i, accs[i].s1, accs[i].s2)
    if world > 1:
        dist.all_reduce(spectra)
    out = spectra.cpu().numpy()
    k = n_components or D
    return [out[i, :k] for i in range(len(accs))]


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

    def _set(self, w, n_components=None):
        """w: full descending spectrum (numpy). n_components defaults to what IncrementalPCA(n_components=None) settles on at
        its first partial_fit: min(samples of the first batch, features) (sklearn _incremental_pca.py)."""
        k = n_components or min(self.first_batch or len(w), len(w))
        mean = getattr(self.acc, "mean_global", None)
        self.mean_ = (mean if mean is not None else self.acc.s1 / self.acc.n).cpu().numpy()
        self.explained_variance_ = w[:k]
        self.explained_variance_ratio_ = w[:k] / w.sum()
        self.n_components_ = k
        self.n_samples_seen_ = self.acc.n
        return self

    def finalize(self, n_components=None):
        return self._set(finalize_head_spectra([self.acc])[0], n_components)


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


def run_PCA(clap, dataloader, num_layers, num_heads, components=None, data_filling="repeatpad", pad_or_truncate=False):
    """src/analyze_attention.py:13-59. Returns {layer: {head: fitted HeadPCA}}."""
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
    for m, w in zip(models, finalize_head_spectra([m.acc for m in models])):   # heads sharded over ranks when distributed
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
