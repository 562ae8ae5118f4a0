"""-m gpu: the ResiDual training step (config c3): backward kernels vs autograd, lambda gradients vs the reference's
loss.backward() (golden) and vs autograd through the oracle.

Tolerances (relative l2 error of each layer's lambda-gradient vector; measured values from tools/train_tol_report.py on B200).
The backward runs on the same bf16 tensor-core GEMMs as the forward, so gradients carry the forward's bf16 error (<= 1e-2,
north_star) plus their own.
* Loss on `embedding` (GELU / LayerNorm / softmax only: smooth): <= 1e-2 against autograd through the fp32 oracle
  (measured 4.9e-3 ... 8.7e-3 over the three cases).
* Zero-shot loss on `audio_embed`, committed golden of the reference's own loss.backward(): measured 8.7e-3 ... 9.7e-3 per layer,
  asserted <= 1.2e-2 (the path crosses the ReLU of audio_projection, model.py:539-543: a bf16-sized perturbation of the 768-d
  embedding flips the gate of the few hidden units that sit within that perturbation of zero, each flip changes the gradient
  discontinuously; the bound leaves 20 % over the measured value rather than the factor 2 it had in round 1).
* The same loss on another seed / a subset of layers (one flipped gate there: element-wise 1.5e-2): direction and norm are
  asserted (cosine > 0.999, measured 0.99989; norm ratio within 1 %, measured 0.998) plus the element-wise bound 2e-2.
"""
import pytest
import torch

import gpu_checks as G

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("C", [96, 128, 192, 384, 768, 1536])
def test_layernorm_bwd(C):
    assert G.check_layernorm_bwd(1000, C) < 1e-5
    assert G.check_layernorm_bwd(333, C, with_add=False) < 1e-5


@pytest.mark.parametrize("B,R,C,nH,shift", [(2, 64, 96, 4, 0), (2, 64, 96, 4, 4), (2, 32, 192, 8, 4), (3, 16, 384, 16, 4),
                                            (2, 8, 768, 32, 4), (2, 64, 128, 4, 4), (2, 16, 512, 16, 0)])
def test_window_attention_bwd(B, R, C, nH, shift):
    dq, dk, dv = G.check_window_attention_bwd(B, R, C, nH, shift)
    assert max(dq, dk, dv) < 5e-3, (dq, dk, dv)     # bf16 outputs: 2^-9 rounding + bf16 P/dS operands


def test_training_step_vs_golden():
    m = G.check_training_step_vs_golden("htsat_tiny_b2.npz")
    assert m["loss_abs"] < 2e-3 and m["sims"] < G.TOL_BF16, m
    for l in range(4):
        assert m[f"lambda_grad{l}"] < 1.2e-2, m


@pytest.mark.parametrize("layers,B,wseed", [((0, 1, 2, 3), 3, 99), ((2, 3), 2, 1234), ((1,), 2, 7)])
def test_embedding_loss_lambda_grads_vs_oracle(layers, B, wseed):
    m = G.check_embedding_grad_vs_oracle("tiny", B, layers, 0, wseed)
    assert m["embedding"] < G.TOL_BF16, m
    for l in layers:
        assert m[f"lambda_grad{l}"] < 1e-2, m


def test_base_model_lambda_grads_vs_oracle():
    """The training step on HTSAT-base (C = 128 ... 1024): `gemm_dual` at K = 128 / 256 ... 1024, the gelu' GEMM pair at C >= 384.
    Same bound as the tiny model's smooth-loss cases."""
    m = G.check_embedding_grad_vs_oracle("base", 2, (0, 1, 2, 3), 0, 321)
    assert m["embedding"] < G.TOL_BF16, m
    for l in range(4):
        assert m[f"lambda_grad{l}"] < 1e-2, m


def test_zero_shot_step_subset_of_layers_vs_oracle():
    m = G.check_training_step_vs_oracle("tiny", 2, (1,), cosine=True)
    assert m["loss_abs"] < 2e-3 and m["sims"] < G.TOL_BF16, m
    assert m["lambda_cos1"] > 0.999 and abs(m["lambda_norm_ratio1"] - 1) < 0.01 and m["lambda_grad1"] < 2e-2, m


@pytest.mark.parametrize("model,env", [("tiny", {}), ("tiny", {"ARD_FUSED_FFN": "0", "ARD_FUSED_FFN_WIDE": "0"}), ("base", {})])
def test_training_forward_equals_bf16_inference(model, env, monkeypatch):
    """The bf16 training forward (tape slots instead of the workspace) computes exactly what bf16 inference does. Inference is
    kept off the fused attention block, which training cannot take (it keeps qkv / ao on chip). The unfused-FFN tiny case and
    HTSAT-base run the patched block's FFN pair on the LayerNorm + GEMM chain at every width."""
    monkeypatch.setenv("ARD_ATTN_BLOCK", "0")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    clap, _, _ = G.make_encoder(model, residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(2, seed=1234).cuda()
    with torch.no_grad():
        ref = enc.encode(waveform=wave, want_audio_embed=True)
        got = enc.encode(waveform=wave, want_audio_embed=True, save_for_backward=True)
        again = enc.encode(waveform=wave, want_audio_embed=True)
    torch.cuda.synchronize()
    for k in ("embedding", "audio_embed"):
        assert torch.equal(got[k], ref[k]), (k, G.rel(got[k], ref[k]))
        assert torch.equal(again[k], ref[k]), k


def test_backward_requires_saved_forward():
    clap, sd, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(1, seed=3).cuda()
    with torch.no_grad():
        enc.encode(waveform=wave)                      # inference forward: nothing saved
    from audio_residual_b200 import lib as L
    import ctypes as C
    a = L.ArdBackwardArgs()
    a.B = 1
    g = torch.zeros(1, enc.num_features, device="cuda")
    a.grad_embedding = g.data_ptr()
    rc = L.load().ard_encoder_backward(enc._hb.h, C.byref(a), L.stream_ptr())
    assert rc == L.ARD_ERR_STATE
    with pytest.raises(RuntimeError):
        L.check(rc)


def test_optimizer_step_changes_output():
    """Adam over the lambdas (src/training.py:106) through the mirror API: the loss decreases over a few steps."""
    clap, sd, _ = G.make_encoder("tiny", residual=True)
    wave = G.W.make_clips(4, seed=21)
    text = G.W.make_text_embeds(50, 512, seed=7)
    labels = torch.tensor([3, 17, 3, 41])
    opt = torch.optim.Adam([r.learnable for r in clap._residuals.values()], lr=0.05)
    losses = []
    for _ in range(4):
        opt.zero_grad()
        loss, _ = G._train_step(clap, wave, text, labels, zero=False)
        opt.step()
        losses.append(loss)
    assert losses[-1] < losses[0], losses
