"""`not gpu`: the oracle (oracle/htsat_oracle.py) against the golden vectors produced by the REAL reference code
(oracle/make_golden.py), and - when /root/reference is mounted - against the reference modules directly."""
import os

import numpy as np
import pytest
import torch

from audio_residual_b200 import weights as W
from oracle import htsat_oracle as O
from oracle import refimport

from gpu_checks import GOLDEN, golden_sample, rel


def _ores(model, seed):
    pca, lam = W.make_pca(model, seed=seed)
    return {l: (torch.tensor(pca[l]["mean"], dtype=torch.float32), torch.tensor(pca[l]["components"], dtype=torch.float32),
                torch.from_numpy(lam[l]).clone().requires_grad_(True)) for l in pca}


@pytest.fixture(scope="module")
def tiny():
    g = np.load(os.path.join(GOLDEN, "htsat_tiny_b2.npz"))
    sd = W.make_state_dict("tiny", seed=int(g["meta_seed"]))
    wave = W.make_clips(int(g["meta_B"]), seed=1234)
    return g, sd, wave


def _check_dict(g, tag, out, emb, tol=2e-5):
    assert rel(out["embedding"], torch.from_numpy(g[f"{tag}_embedding"])) < tol
    assert rel(emb, torch.from_numpy(g[f"{tag}_audio_embed"])) < tol
    assert rel(out["clipwise_output"], torch.from_numpy(g[f"{tag}_clipwise_output"])) < tol
    assert rel(golden_sample(out["framewise_output"]), torch.from_numpy(g[f"{tag}_framewise_sample"])) < tol
    assert rel(golden_sample(out["fine_grained_embedding"]), torch.from_numpy(g[f"{tag}_fine_sample"])) < tol
    for l in range(4):
        assert rel(golden_sample(out["layers_residuals"][l]), torch.from_numpy(g[f"{tag}_res{l}_sample"])) < tol
        assert rel(golden_sample(out["layers_attention"][l]), torch.from_numpy(g[f"{tag}_attn{l}_sample"])) < tol
        r = out["layers_residuals"][l].double()
        cks = np.array([r.sum().item(), r.abs().sum().item(), (r * r).sum().item()])
        assert np.allclose(cks[1:], g[f"{tag}_res{l}_cks"][1:], rtol=1e-4)


def test_oracle_plain_vs_golden(tiny):
    g, sd, wave = tiny
    with torch.no_grad():
        out = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["tiny"])
        emb = O.audio_projection(out["embedding"], sd)
    _check_dict(g, "plain", out, emb)
    lm = O.logmel(O.stft_power(wave, sd), sd)
    assert rel(golden_sample(lm), torch.from_numpy(g["logmel_sample"])) < 1e-5
    img = O.reshape_wav2img(O.bn0_eval(lm, sd))
    assert rel(golden_sample(img), torch.from_numpy(g["img_sample"])) < 1e-5
    assert rel(golden_sample(O.patch_embed(img, sd)), torch.from_numpy(g["patch_embed_sample"])) < 1e-5
    # the bicubic time resize leaves frequency untouched and folds time into 4 stacked quarters (SURVEY §0.3)
    x = O.bn0_eval(lm, sd)
    xi = torch.nn.functional.interpolate(x, (1024, 64), mode="bicubic", align_corners=True)
    assert torch.equal(img[:, 0, 64 * 2 + 5, :], xi[:, 0, 2 * 256:3 * 256, 5])


def test_oracle_residual_and_grads_vs_golden(tiny):
    g, sd, wave = tiny
    ores = _ores("tiny", int(g["meta_seed"]))
    out = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["tiny"], ores)
    emb = O.audio_projection(out["embedding"], sd)
    with torch.no_grad():
        _check_dict(g, "residual", {k: (v.detach() if torch.is_tensor(v) else [t.detach() for t in v]) for k, v in out.items()}, emb.detach())
    text = W.make_text_embeds(50, 512, seed=7)
    labels = torch.from_numpy(g["labels"])
    sims = emb @ text.T
    loss = torch.nn.functional.cross_entropy(sims, labels)
    loss.backward()
    assert abs(loss.item() - float(g["train_loss"])) < 1e-5
    assert rel(sims.detach(), torch.from_numpy(g["train_sims"])) < 2e-5
    for l in range(4):
        assert rel(ores[l][2].grad, torch.from_numpy(g[f"lambda_grad{l}"])) < 5e-4
    # linear probe head (src/linear.py:23-45)
    Wc = torch.from_numpy(g["cls_weight"]).requires_grad_(True)
    bc = torch.zeros(50, requires_grad=True)
    logits = torch.nn.functional.linear(emb.detach(), Wc, bc)
    l2 = torch.nn.functional.cross_entropy(logits, labels)
    l2.backward()
    assert abs(l2.item() - float(g["cls_loss"])) < 1e-5
    assert rel(Wc.grad, torch.from_numpy(g["cls_weight_grad"])) < 1e-4 and rel(bc.grad, torch.from_numpy(g["cls_bias_grad"])) < 1e-4


def test_oracle_base_fusion_vs_golden():
    g = np.load(os.path.join(GOLDEN, "htsat_base_fusion_b2.npz"))
    sd = W.make_state_dict("base", seed=int(g["meta_seed"]))
    wave = W.make_clips(int(g["meta_B"]), seed=1234)
    fb = torch.from_numpy(W.mel_filterbank(htk=True, slaney_norm=False)).float()
    win = torch.from_numpy(W.hann_periodic(1024)).float()
    mel = torch.stack([O.fusion_mel(w, fb, win) for w in wave])
    mf = torch.stack([mel] * 4, dim=1)
    assert rel(golden_sample(mf), torch.from_numpy(g["mel_fusion_sample"])) < 1e-5     # torchaudio get_mel (data.py:363-399)
    with torch.no_grad():
        out = O.htsat_forward({"mel_fusion": mf}, sd, O.CONFIGS["base"], enable_fusion=True)
        emb = O.audio_projection(out["embedding"], sd)
    _check_dict(g, "plain", out, emb, tol=5e-5)


def test_oracle_base_waveform_route_vs_golden():
    """HTSAT-base without feature fusion (C = 128 ... 1024, head dim 32), plain and with ResiDual on all layers, against what the
    real reference produced (oracle/make_golden.py run_case("base", False, ...))."""
    g = np.load(os.path.join(GOLDEN, "htsat_base_b2.npz"))
    seed = int(g["meta_seed"])
    sd = W.make_state_dict("base", seed=seed)
    wave = W.make_clips(int(g["meta_B"]), seed=1234)
    with torch.no_grad():
        out = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["base"])
        _check_dict(g, "plain", out, O.audio_projection(out["embedding"], sd), tol=5e-5)
        ores = {l: (mu, comp, lam.detach()) for l, (mu, comp, lam) in _ores("base", seed).items()}
        out = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["base"], ores)
        _check_dict(g, "residual", out, O.audio_projection(out["embedding"], sd), tol=5e-5)


def test_quantize_and_padding():
    x = torch.tensor([-1.5, -1.0, -0.5, 0.0, 1e-5, 0.3333, 0.99999, 1.0, 2.0])
    q = O.quantize_tensor(x)
    assert torch.equal(q, torch.from_numpy(O.int16_roundtrip_np(x.numpy())))
    assert q.min() == -1.0 and q.max() == 1.0 and q[3] == 0.0
    assert torch.equal(O.quantize_tensor(q), q)                      # idempotent
    w = torch.arange(5, dtype=torch.float32)
    assert O.pad_clip(w, 12, "repeatpad").tolist() == [0, 1, 2, 3, 4, 0, 1, 2, 3, 4, 0, 0]
    assert O.pad_clip(w, 12, "pad").tolist() == [0, 1, 2, 3, 4] + [0] * 7
    assert O.pad_clip(w, 12, "repeat").tolist() == [0, 1, 2, 3, 4, 0, 1, 2, 3, 4, 0, 1]
    assert O.pad_clip(w, 5).tolist() == [0, 1, 2, 3, 4]
    with pytest.raises(NotImplementedError):
        O.pad_clip(w, 12, "bogus")
    with pytest.raises(AttributeError):
        O.pad_clip(torch.zeros(13), 12)


def test_pca_from_moments_vs_incremental_pca_golden():
    g = np.load(os.path.join(GOLDEN, "pca_moments.npz"))
    got = O.pca_from_moments(int(g["n"]), g["s1"], g["s2"])
    assert np.allclose(got["mean"], g["mean"], atol=1e-6)
    assert np.allclose(got["explained_variance"], g["explained_variance"], rtol=2e-5)
    assert np.allclose(got["explained_variance_ratio"], g["explained_variance_ratio"], rtol=2e-5)
    assert np.allclose(got["components"], g["components"], atol=5e-6)
    pr, idim = O.spectrum_summaries(got["explained_variance"], got["explained_variance_ratio"])
    assert 1.0 <= pr <= 96 and 1 <= idim <= 96


def test_residual_identities():
    """ResiDual quirks the drop-in must keep (SURVEY Q1, Q11): no '+ mean'; with lambda=1 and a full orthonormal basis the
    module returns x - mean; the fold used by the CUDA path (W' = M W, b' = (b - mean) M) is exact algebra."""
    torch.manual_seed(0)
    D = 96
    q, _ = torch.linalg.qr(torch.randn(D, D, dtype=torch.float64))
    mean = torch.randn(D, dtype=torch.float64)
    x = torch.randn(7, 5, D, dtype=torch.float64)
    assert torch.allclose(O.residual_apply(x, mean, q.T, torch.ones(D, dtype=torch.float64)), x - mean, atol=1e-12)
    lam = 1 + 0.1 * torch.randn(D, dtype=torch.float64)
    Wp, bp = torch.randn(D, D, dtype=torch.float64), torch.randn(D, dtype=torch.float64)
    a = torch.randn(11, D, dtype=torch.float64)
    ref = O.residual_apply(a @ Wp.T + bp, mean, q.T, lam)
    M = q @ torch.diag(lam) @ q.T          # = B^T diag(lam) B with B = q.T
    assert torch.allclose(a @ (M @ Wp).T + (bp - mean) @ M, ref, atol=1e-10)


@pytest.mark.skipif(not refimport.available(), reason="needs the reference sources (ARD_REFERENCE_ROOT or oracle/_ref), not stored in this repository")
def test_oracle_block_vs_live_reference():
    """Direct op-level pin against the imported reference modules, where their sources are available. Without them the oracle stays
    pinned to the reference by the goldens it produced (test_oracle_*_vs_golden above: every block's residual and attention output of
    HTSAT-tiny / -base, plain and ResiDual-patched, and the ResiDual module's autograd)."""
    ns = refimport.load()
    torch.manual_seed(3)
    blk = ns.htsat.SwinTransformerBlock(dim=96, input_resolution=(16, 16), num_heads=4, window_size=8, shift_size=4).eval()
    for p in blk.parameters():
        torch.nn.init.normal_(p, std=0.2)
    sd = {"layers.0.blocks.0." + k: v for k, v in blk.state_dict().items()}
    x = torch.randn(2, 256, 96)
    with torch.no_grad():
        r_x, r_attn, r_res = blk(x)
        o_x, o_attn, o_res = O.swin_block(x, sd, "layers.0.blocks.0.", 16, 16, 4, 4)
    assert rel(o_x, r_x) < 1e-6 and rel(o_attn, r_attn) < 1e-6 and rel(o_res, r_res) < 1e-6
    res = ns.residual.ResiDual(torch.linalg.qr(torch.randn(96, 96))[0].T.contiguous(), 0.1 * torch.randn(96))
    with torch.no_grad():
        res.learnable.copy_(1 + 0.1 * torch.randn(96))
    ns.residual.patch_block_with_residual(blk, res)
    with torch.no_grad():
        r_x, r_attn, r_res = blk(x)
        o_x, o_attn, o_res = O.swin_block(x, sd, "layers.0.blocks.0.", 16, 16, 4, 4, (res.mean, res.basis, res.learnable))
    assert rel(o_x, r_x) < 1e-6 and rel(o_res, r_res) < 1e-6


def test_oracle_head_outputs_and_residual_module_vs_reference_golden():
    """Round-2 goldens (oracle/make_golden_extras.py): the per-head `attn @ v` tap obtained by hooking the real reference, the
    reference ResiDual module's autograd, and ResiDual on layers (0, 2) with truncated bases."""
    g = np.load(os.path.join(GOLDEN, "extras_tiny_b2.npz"))
    sd = W.make_state_dict("tiny", seed=int(g["meta_seed"]))
    wave = W.make_clips(int(g["meta_B"]), seed=1234)
    with torch.no_grad():
        out = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["tiny"], None, head_outputs=True)
    for l in range(4):
        t = out["head_outputs"][l]
        assert tuple(t.shape) == tuple(g[f"head_out{l}_shape"])
        assert rel(golden_sample(t), torch.from_numpy(g[f"head_out{l}_sample"])) < 2e-5
    x = torch.from_numpy(g["residual_module_x"]).requires_grad_(True)
    lam = torch.from_numpy(g["residual_module_lam"][:40].copy()).requires_grad_(True)
    y = O.residual_apply(x, torch.from_numpy(g["residual_module_mean"]), torch.from_numpy(g["residual_module_basis"][:40]), lam)
    y.backward(torch.from_numpy(g["residual_module_gout"]))
    assert rel(y.detach(), torch.from_numpy(g["residual_module_k40_out"])) < 1e-6
    assert rel(x.grad, torch.from_numpy(g["residual_module_k40_dx"])) < 1e-6
    assert rel(lam.grad, torch.from_numpy(g["residual_module_k40_dlam"])) < 1e-5
    pca, lm = W.make_pca("tiny", seed=int(g["meta_seed"]))
    ores = {int(l): (torch.tensor(pca[int(l)]["mean"], dtype=torch.float32), torch.tensor(pca[int(l)]["components"][:int(k)], dtype=torch.float32),
                     torch.from_numpy(lm[int(l)][:int(k)].copy())) for l, k in zip(g["subset_layers"], g["subset_k"])}
    with torch.no_grad():
        sub = O.htsat_forward({"waveform": wave}, sd, O.CONFIGS["tiny"], ores)
    assert rel(sub["embedding"], torch.from_numpy(g["subset_embedding"])) < 2e-5
    for l in range(4):
        assert rel(golden_sample(sub["layers_residuals"][l]), torch.from_numpy(g[f"subset_res{l}_sample"])) < 2e-5
