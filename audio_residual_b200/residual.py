"""Mirror of the reference's src/residual.py on top of libard_b200.so.

Same public names and argument meaning: ResiDual, patch_block_with_residual, setup_residual_htsat, load_residual,
compute_pca_components, quantize_tensor, pad_or_truncate. Differences are only in where the arithmetic runs:

* ResiDual's centre-project-scale-reproject (src/residual.py:29-42) is folded, for the current lambda, into the attention
  out-projection of every patched block (W' = M W_proj, b' = (b_proj - mean) M, M = B^T diag(lambda) B) inside the C
  library, so it costs no extra pass over the tokens; the patched block keeps the reference's doubled shortcut/FFN
  (src/residual.py:91-96).
* compute_pca_components accumulates {n, sum x, sum x x^T} on the GPU and eigendecomposes once, which is what
  IncrementalPCA(n_components=None) converges to (SURVEY.md §0.3); the pickle schema is unchanged.
"""
import copy
import ctypes as C
import os
import pickle

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import lib as L


class ResiDual(nn.Module):
    """src/residual.py:14-42. Buffers `mean` [D], `basis` [K, D]; parameter `learnable` [K] initialised to ones."""

    def __init__(self, pca_basis, pca_mean, n_components=None):
        super().__init__()
        D = pca_basis.shape[0]
        self.n_components = n_components or D
        self.register_buffer("mean", pca_mean)
        self.register_buffer("basis", pca_basis[:self.n_components])
        self.learnable = nn.Parameter(torch.ones(self.n_components))

    def forward(self, x):
        """x [B, N, D] (CUDA) -> ((x - mean) @ basis.T * learnable) @ basis   (src/residual.py:29-42; the mean is not re-added).
        Differentiable in `x` and in `learnable` like the reference module (autograd node = ard_residual_forward /
        ard_residual_backward: bf16 tcgen05 GEMMs, lambda-gradient reduced in the kernel)."""
        if not x.is_cuda:
            raise RuntimeError("audio_residual_b200.ResiDual runs on CUDA only (no CPU fallback)")
        dev = x.device
        return _ResiDualFn.apply(x, self.learnable, self.mean.to(dev), self.basis.to(dev))   # the reference re-copies per call too (Q4)


class _ResiDualFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, lam, mean, basis):
        dev = x.device
        D = x.shape[-1]
        x2 = x.detach().to(torch.float32).contiguous().view(-1, D)
        lam_d = lam.detach().to(dev, torch.float32).contiguous()
        mean_d = mean.detach().to(dev, torch.float32).contiguous()
        basis_d = basis.detach().to(dev, torch.float32).contiguous()
        K = basis_d.shape[0]
        if basis_d.shape[1] != D or mean_d.numel() != D or lam_d.numel() != K:
            raise ValueError(f"ResiDual: x has width {D}, basis {tuple(basis_d.shape)}, mean {tuple(mean_d.shape)}, learnable {tuple(lam_d.shape)}")
        out = torch.empty_like(x2)
        with torch.cuda.device(dev):
            L.check(L.load().ard_residual_forward(L.ptr(x2), L.ptr(mean_d), L.ptr(basis_d), L.ptr(lam_d), L.ptr(out), x2.shape[0], D, K,
                                                  L.stream_ptr()))
        ctx.save_for_backward(x2, lam_d, mean_d, basis_d)
        ctx.xshape, ctx.lam_dev, ctx.lam_dtype = x.shape, lam.device, lam.dtype
        return out.view(x.shape)

    @staticmethod
    def backward(ctx, g):
        x2, lam_d, mean_d, basis_d = ctx.saved_tensors
        dev = x2.device
        rows, D = x2.shape
        K = basis_d.shape[0]
        g2 = g.detach().to(dev, torch.float32).contiguous().view(-1, D)
        dx = torch.empty_like(x2) if ctx.needs_input_grad[0] else None
        dlam = torch.zeros(K, device=dev, dtype=torch.float32) if ctx.needs_input_grad[1] else None
        with torch.cuda.device(dev):
            L.check(L.load().ard_residual_backward(L.ptr(x2), L.ptr(g2), L.ptr(mean_d), L.ptr(basis_d), L.ptr(lam_d), L.ptr(dx), L.ptr(dlam),
                                                   rows, D, K, L.stream_ptr()))
        return (dx.view(ctx.xshape) if dx is not None else None,
                dlam.to(ctx.lam_dev, ctx.lam_dtype) if dlam is not None else None, None, None)


def patch_block_with_residual(block, residual):
    """src/residual.py:45-100: inject `residual` after the block's attention. The block's forward keeps returning
    (x, attn, residual_x) with residual_x the POST-ResiDual tensor, and reproduces the doubled shortcut/FFN.
    As in the reference the ResiDual is referenced, not registered: it does not appear in model.parameters()."""
    object.__setattr__(block, "_residual", residual)


def load_residual(pca_path):
    """src/residual.py:161-174"""
    with open(pca_path, "rb") as f:
        pca_results = pickle.load(f)
    basis = torch.tensor(pca_results["components"], dtype=torch.float32)
    mean = torch.tensor(pca_results["mean"], dtype=torch.float32)
    return ResiDual(basis, mean)


def setup_residual_htsat(model, pca_files, layers):
    """src/residual.py:176-207: deep-copy the encoder, freeze it, load one ResiDual per listed layer (shared by all the
    layer's blocks, so lambda-gradients sum over blocks), leave only `learnable` trainable."""
    model = copy.deepcopy(model)
    for p in model.parameters():
        p.requires_grad = False
    residuals = {}
    for l in layers:
        if l >= len(model.layers):
            raise ValueError(f"Layer index {l} out of range for model with {len(model.layers)} layers")
        res = load_residual(pca_files[l])
        for p in res.parameters():
            p.requires_grad = False
        res.learnable.requires_grad = True
        residuals[l] = res
    for l in layers:
        for b in range(len(model.layers[l].blocks)):
            patch_block_with_residual(model.layers[l].blocks[b], residuals[l])
    return model, residuals


def inject_residuals(model, pca, lambdas=None):
    """Convenience used by bench/smoke: patch `model` IN PLACE from in-memory PCA dicts {layer: {"components", "mean"}}."""
    residuals = {}
    for l, d in pca.items():
        res = ResiDual(torch.tensor(d["components"], dtype=torch.float32), torch.tensor(d["mean"], dtype=torch.float32))
        if lambdas is not None:
            with torch.no_grad():
                res.learnable.copy_(torch.as_tensor(lambdas[l], dtype=torch.float32))
        residuals[l] = res
        for blk in model.layers[l].blocks:
            patch_block_with_residual(blk, res)
    return residuals


def save_lambdas(residuals, path):
    """The reference never persists the trained `learnable` vectors (the ResiDual modules are not registered on the model,
    SURVEY Q4); this writes {layer: lambda[K]} so a trained reweighting can be restored with load_lambdas."""
    torch.save({int(l): r.learnable.detach().cpu().clone() for l, r in residuals.items()}, path)


def load_lambdas(residuals, path):
    sd = torch.load(path, map_location="cpu")
    for l, r in residuals.items():
        if int(l) not in sd:
            raise KeyError(f"no lambda saved for layer {l}")
        if sd[int(l)].shape != r.learnable.shape:
            raise ValueError(f"layer {l}: saved lambda has shape {tuple(sd[int(l)].shape)}, expected {tuple(r.learnable.shape)}")
        with torch.no_grad():
            r.learnable.copy_(sd[int(l)].to(r.learnable.device))
    return residuals


def quantize_tensor(audio_tensor: torch.Tensor) -> torch.Tensor:
    """src/residual.py:210-212 (runs on the tensor's device; a fused on-device variant is `quantize=True` on the encoder)."""
    audio_tensor = torch.clamp(audio_tensor, -1.0, 1.0)
    return (audio_tensor * 32767.0).to(torch.int16).to(torch.float32) / 32767.0


def pad_or_truncate(audio_tensor, target_len=480000):
    """src/residual.py:214-222"""
    if audio_tensor.dim() > 1:
        audio_tensor = audio_tensor.mean(dim=0)
    length = audio_tensor.shape[0]
    if length > target_len:
        return audio_tensor[:target_len]
    elif length < target_len:
        return F.pad(audio_tensor, (0, target_len - length), mode="constant")
    return audio_tensor


class MomentAccumulator:
    """{n, sum x, sum x x^T} in float64 on the GPU (ard_stats_accumulate); `allreduce()` sums them over ranks.

    Wide accumulators (the 4096-d attention maps) park short batches of rows in a device buffer and run the X^T X GEMM + float64
    fold once `min_rows` of them are there: the fold moves the whole D x D accumulator (64 MB fp32 G + 128 MB float64 for D = 4096)
    whatever the row count, so the last layer's 32 heads with one window per clip (128 rows per step at B = 128) paid it for a
    GEMM of 0.1 ms. `s1` / `s2` flush the parked rows before they are read, so callers always see exact moments."""

    def __init__(self, D, device, min_rows=None):
        self.D, self.n = D, 0
        self._s1 = torch.zeros(D, device=device, dtype=torch.float64)
        self._s2 = torch.zeros(D, D, device=device, dtype=torch.float64)
        self.min_rows = (2048 if D >= 2048 else 0) if min_rows is None else int(min_rows)
        self._buf, self._fill = None, 0

    @property
    def s1(self):
        self.flush()
        return self._s1

    @s1.setter
    def s1(self, v):
        self._s1 = v

    @property
    def s2(self):
        self.flush()
        return self._s2

    @s2.setter
    def s2(self, v):
        self._s2 = v

    def _accumulate(self, x2, ldx):
        with torch.cuda.device(x2.device):
            L.check(L.load().ard_stats_accumulate_strided(C.c_void_p(x2.data_ptr()), x2.shape[0], ldx, self.D, L.ptr(self._s1), L.ptr(self._s2),
                                                          L.stream_ptr()))

    def flush(self):
        if self._fill:
            self._accumulate(self._buf[:self._fill], self.D)
            self._fill = 0
            self._flushed = True

    def parked_rows(self):
        """The samples themselves, [n, D] fp32, while every one of them is still parked (nothing folded into s2 yet), else None.
        With fewer samples than dimensions the covariance spectrum is the spectrum of the n x n Gram matrix of the centred rows:
        analyze_attention.finalize_head_spectra takes that route instead of a D x D eigen-solve."""
        if getattr(self, "_flushed", False) or self._buf is None or self._fill != self.n:
            return None
        return self._buf[:self._fill]

    def update(self, x):
        x = x.detach()
        if x.dim() == 2 and x.dtype == torch.float32 and x.stride(1) == 1 and x.shape[1] == self.D and x.stride(0) >= self.D:
            x2, ldx = x, x.stride(0)          # a strided row view (one head's maps) is read in place
        else:
            x2 = x.to(torch.float32).contiguous().view(-1, self.D)
            ldx = self.D
        rows = x2.shape[0]
        self.n += rows
        if rows >= self.min_rows:
            self.flush()
            self._accumulate(x2, ldx)
            self._flushed = True
            return
        if self._buf is None:
            self._buf = torch.empty(self.min_rows, self.D, device=self._s1.device, dtype=torch.float32)
        if self._fill + rows > self.min_rows:
            self.flush()
        self._buf[self._fill:self._fill + rows].copy_(x2)
        self._fill += rows
        if self._fill == self.min_rows:
            self.flush()

    def allreduce(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            n = torch.tensor([self.n], device=self.s1.device, dtype=torch.float64)
            dist.all_reduce(n)
            dist.all_reduce(self.s1)
            dist.all_reduce(self.s2)
            self.n = int(n.item())
        return self

    def pca(self, n_components=None):
        """PCA dict (pca_from_moments' schema) of the moments. On a CUDA accumulator the covariance is assembled and solved on the
        device (pca_on_device); on the CPU it goes through pca_from_moments."""
        if self._s1.device.type == "cuda":
            return pca_on_device(self.n, self.s1, self.s2, n_components)
        return pca_from_moments(self.n, self.s1.cpu().numpy(), self.s2.cpu().numpy(), n_components)


def pca_from_moments(n, s1, s2, n_components=None):
    """PCA dict in the reference pickle schema (src/residual.py:143-150) from the sufficient statistics. Matches
    sklearn IncrementalPCA(n_components=None) on full-rank data: ddof=1 variances, components sorted by decreasing
    variance, sign fixed by svd_flip(u_based_decision=False) (largest-|entry| of each row positive)."""
    s1 = np.asarray(s1, dtype=np.float64)
    s2 = np.asarray(s2, dtype=np.float64)
    mean = s1 / n
    cov = (s2 - n * np.outer(mean, mean)) / (n - 1)
    cov = 0.5 * (cov + cov.T)
    w, v = np.linalg.eigh(cov)
    order = np.argsort(w)[::-1]
    w = np.maximum(w[order], 0.0)
    comps = v[:, order].T
    idx = np.argmax(np.abs(comps), axis=1)
    signs = np.sign(comps[np.arange(comps.shape[0]), idx])
    signs[signs == 0] = 1.0
    comps = comps * signs[:, None]
    total = w.sum()
    k = n_components or comps.shape[0]
    return {"components": comps[:k], "mean": mean, "explained_variance": w[:k], "explained_variance_ratio": w[:k] / total,
            "n_components": k, "input_dim": comps.shape[1], "num_samples": int(n)}


def pca_on_device(n, s1, s2, n_components=None):
    """pca_from_moments for float64 moments on a CUDA device: the ddof=1 covariance is assembled there and solved there, by
    ard_sym_eigh or torch.linalg.eigh, whichever was measured faster at this width (linalg.eigh_batch); ordering, clamping, the
    sign rule and the truncation to n_components (from the one solve) are pca_from_moments'. Returns the same dict of numpy float64
    arrays."""
    from .linalg import eigh_batch, sign_fix
    mean = s1 / n
    cov = (s2 - n * torch.outer(mean, mean)) / (n - 1)
    cov = 0.5 * (cov + cov.t())
    w, Q = eigh_batch(cov[None])
    w, Q = w[0], Q[0]
    k = n_components or cov.shape[0]
    comps = sign_fix(Q.mT.flip(0)[:k])
    w = w.flip(0).clamp_min(0).cpu().numpy()
    total = w.sum()
    return {"components": comps.cpu().numpy(), "mean": mean.cpu().numpy(), "explained_variance": w[:k],
            "explained_variance_ratio": w[:k] / total, "n_components": k, "input_dim": cov.shape[0], "num_samples": int(n)}


def compute_pca_components(model, dataloader, target_layer, n_components=None, max_batches=None, save_path=None, max_len=480000,
                           data_filling="repeatpad", pad_or_truncate=False):
    """src/residual.py:103-159. `model` is the CLAP_Module wrapper; batches are (waveform[B,1,T], ...)."""
    from .clap import batch_features
    model.eval()
    acc = None
    enc = model.model.audio_branch
    if not 0 <= target_layer < enc.num_layers:
        raise IndexError(f"target_layer {target_layer} out of range for a model with {enc.num_layers} layers")   # src/residual.py:135 (list index)
    with torch.no_grad():                                      # src/residual.py:118
        for i, batch in enumerate(dataloader):
            if max_batches and i >= max_batches:
                break
            x = batch[0]
            feats = batch_features(x.squeeze(1), max_len, data_filling, device=model.device, do_pad_or_truncate=pad_or_truncate)
            out = enc.encode(waveform=feats, quantize=True, want_dict=True) if not enc.enable_fusion else \
                enc.encode(mel_fusion=model.fusion_mel(feats, quantize=True), want_dict=True)
            res = out["layers_residuals"][target_layer]
            if acc is None:
                acc = MomentAccumulator(res.shape[-1], res.device)
            acc.update(res)
    if acc is None:
        raise ValueError("compute_pca_components: the dataloader produced no batch")
    pca_results = acc.allreduce().pca(n_components)
    if save_path:
        os.makedirs(os.path.dirname(save_path), exist_ok=True)
        with open(save_path, "wb") as f:
            pickle.dump(pca_results, f)
        print(f"PCA results saved to {save_path}")
    return pca_results
