"""-m gpu: the fp32-grade training step (encoder.train_precision = "fp32"): fp32 tape, 3-term split-bf16 dgrads on tcgen05,
fp32 window-attention / gelu' / LayerNorm backward. Tolerances are the fp32 tier (G.TOL_FP32 = 1e-4, rel. l2 error) against
the reference's own fp32 loss.backward() (golden) and against autograd through the fp32 oracle.
"""
import copy
import ctypes as C

import pytest
import torch

import gpu_checks as G
from audio_residual_b200 import lib as L

pytestmark = pytest.mark.gpu


@pytest.fixture
def fp32_training(monkeypatch):
    """Every encoder the shared check flows build trains at fp32 grade."""
    make = G.make_encoder

    def make_fp32(*a, **k):
        clap, sd, ores = make(*a, **k)
        clap.model.audio_branch.train_precision = "fp32"
        return clap, sd, ores

    monkeypatch.setattr(G, "make_encoder", make_fp32)


def _attention_f32_bwd(B, R, Cdim, nH, shift, seed=0):
    """ard_window_attention_f32_bwd vs float64 autograd through the oracle's attention core on the same fp32 qkv / dout."""
    g = torch.Generator().manual_seed(seed)
    hd = Cdim // nH
    qkv = torch.randn(B * R * R, 3 * Cdim, generator=g)
    qkv[:, :Cdim] *= hd ** -0.5
    table = 0.5 * torch.randn(225, nH, generator=g)
    dout = torch.randn(B * R * R, Cdim, generator=g)
    qr = qkv.double().requires_grad_(True)
    out, _ = G._ref_window_attention(qr, table.double(), B, R, Cdim, nH, shift)
    out.backward(dout.double())
    qd, dd, td = qkv.cuda(), dout.cuda(), table.cuda()
    dq = torch.zeros(B * R * R, 3 * Cdim, device="cuda")
    L.check(L.load().ard_window_attention_f32_bwd(L.ptr(qd), L.ptr(dd), L.ptr(dq), L.ptr(td), B, R, R, Cdim, nH, shift, L.stream_ptr()))
    torch.cuda.synchronize()
    got, ref = dq.cpu().double(), qr.grad
    return tuple(G.rel(got[:, i * Cdim:(i + 1) * Cdim], ref[:, i * Cdim:(i + 1) * Cdim]) for i in range(3))


@pytest.mark.parametrize("B,R,C,nH,shift", [(2, 64, 96, 4, 0), (2, 64, 96, 4, 4), (2, 32, 192, 8, 4), (3, 16, 384, 16, 4),
                                            (2, 8, 768, 32, 4), (2, 64, 128, 4, 4), (2, 16, 512, 16, 0)])
def test_window_attention_f32_bwd(B, R, C, nH, shift):
    dq, dk, dv = _attention_f32_bwd(B, R, C, nH, shift)
    assert max(dq, dk, dv) < 1e-5, (dq, dk, dv)


def test_training_step_vs_golden_fp32(fp32_training):
    m = G.check_training_step_vs_golden("htsat_tiny_b2.npz")
    assert m["loss_abs"] < 1e-5 and m["sims"] < G.TOL_FP32, m
    for l in range(4):
        assert m[f"lambda_grad{l}"] < G.TOL_FP32, m


@pytest.mark.parametrize("model,layers,B,wseed", [("tiny", (0, 1, 2, 3), 3, 99), ("tiny", (2, 3), 2, 1234), ("tiny", (1,), 2, 7),
                                                  ("base", (0, 1, 2, 3), 2, 321)])
def test_embedding_loss_lambda_grads_vs_oracle_fp32(fp32_training, model, layers, B, wseed):
    m = G.check_embedding_grad_vs_oracle(model, B, layers, 0, wseed)
    assert m["embedding"] < G.TOL_FP32, m
    for l in layers:
        assert m[f"lambda_grad{l}"] < G.TOL_FP32, m


def test_zero_shot_step_subset_of_layers_vs_oracle_fp32(fp32_training):
    """The case with a ReLU gate of audio_projection flipped by the bf16 forward error: at fp32 grade it matches element-wise."""
    m = G.check_training_step_vs_oracle("tiny", 2, (1,))
    assert m["loss_abs"] < 1e-5 and m["sims"] < G.TOL_FP32, m
    assert m["lambda_grad1"] < G.TOL_FP32, m


def test_training_forward_equals_fp32_inference():
    """The fp32-grade training forward (tape slots instead of the workspace) computes exactly what the fp32-grade inference does."""
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(2, seed=1234).cuda()
    with torch.no_grad():
        ref = enc.encode(waveform=wave, want_audio_embed=True, precision="fp32")
        got = enc.encode(waveform=wave, want_audio_embed=True, precision="fp32", save_for_backward=True)
        again = enc.encode(waveform=wave, want_audio_embed=True, precision="fp32")
    torch.cuda.synchronize()
    for k in ("embedding", "audio_embed"):
        assert torch.equal(got[k], ref[k]), (k, G.rel(got[k], ref[k]))
        assert torch.equal(again[k], ref[k]), k


def _lambda_grads(clap, wave, text, labels):
    G._train_step(clap, wave, text, labels)
    return torch.cat([r.learnable.grad.detach().cpu().flatten() for _, r in sorted(clap._residuals.items())])


def test_no_cross_talk_between_precisions():
    """A bf16 step on a handle that just ran an fp32-grade step gives the bf16 step of a fresh handle (to within the spread of
    two bf16 runs there: the lambda reductions use float atomics)."""
    wave = G.W.make_clips(2, seed=1234)
    text = G.W.make_text_embeds(50, 512, seed=7)
    labels = torch.tensor([3, 17])
    fresh, _, _ = G.make_encoder("tiny", residual=True)
    g1 = _lambda_grads(fresh, wave, text, labels)
    g2 = _lambda_grads(fresh, wave, text, labels)
    spread = G.rel(g2, g1)
    used, _, _ = G.make_encoder("tiny", residual=True)
    enc = used.model.audio_branch
    enc.train_precision = "fp32"
    g32 = _lambda_grads(used, wave, text, labels)
    enc.train_precision = "bf16"
    g = _lambda_grads(used, wave, text, labels)
    assert G.rel(g, g1) <= max(2 * spread, 1e-5), (G.rel(g, g1), spread)
    assert torch.isfinite(g32).all() and G.rel(g32, g1) > 1e-5   # the fp32-grade step really ran in between


def test_backward_of_older_fp32_forward_is_refused():
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(1, seed=3).cuda()
    with torch.no_grad():
        gen32 = enc.encode(waveform=wave, precision="fp32", save_for_backward=True)["_tape_generation"]
        gen16 = enc.encode(waveform=wave, save_for_backward=True)["_tape_generation"]
    assert gen16 != gen32
    lib = L.load()
    a = L.ArdBackwardArgs()
    a.B = 1
    g = torch.zeros(1, enc.num_features, device="cuda")
    a.grad_embedding = g.data_ptr()
    dl = [torch.zeros(int(r.learnable.shape[0]), device="cuda") for _, r in sorted(clap._residuals.items())]
    for l, t in zip(sorted(clap._residuals), dl):
        a.grad_lambda[l] = t.data_ptr()
    a.generation = gen32
    assert lib.ard_encoder_backward(enc._hb.h, C.byref(a), L.stream_ptr()) == L.ARD_ERR_STATE
    a.generation = gen16
    L.check(lib.ard_encoder_backward(enc._hb.h, C.byref(a), L.stream_ptr()))
    torch.cuda.synchronize()


def test_optimizer_step_fp32_lowers_loss():
    """Adam over the lambdas (src/training.py:106) through get_audio_embedding_from_data at fp32 grade."""
    clap, _, _ = G.make_encoder("tiny", residual=True)
    clap.model.audio_branch.train_precision = "fp32"
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


def test_train_precision_attribute():
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    assert enc.train_precision == "bf16"
    with pytest.raises(ValueError):
        enc.train_precision = "fp16"
    wave = G.W.make_clips(2, seed=1234).cuda()
    enc.precision = "fp32"                                  # fp32 inference alone does not make the training step fp32
    with pytest.raises(NotImplementedError, match="train_precision"):
        with torch.enable_grad():
            clap.get_audio_embedding_from_data(wave, use_tensor=True)
    enc.train_precision = "fp32"
    with torch.enable_grad():
        emb = clap.get_audio_embedding_from_data(wave, use_tensor=True)
    assert emb.requires_grad
    from audio_residual_b200.residual import setup_residual_htsat
    assert copy.deepcopy(enc).train_precision == "fp32"
    assert setup_residual_htsat(enc, {}, [])[0].train_precision == "fp32"
