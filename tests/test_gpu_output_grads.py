"""-m gpu: gradients into the ResiDual lambdas from every differentiable key of the HTSAT output dict (htsat.py:797-832):
the tail backward (tscam head + fine-grained embedding) and the window-attention backward with a probability gradient at op
level against float64 autograd, lambda gradients per key against
autograd through the oracle (bf16 tier 1e-2 vs the fp32 oracle, fp32-grade tier 1e-4 vs the float64 oracle), reachability of
the lambdas, linearity over keys, the unchanged embedding-loss step, and the error paths of the C ABI.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import gpu_checks as G
from audio_residual_b200 import lib as L

pytestmark = pytest.mark.gpu

O = G.O


# ---------------------------------------------------------------------------------------------------- op level: tail backward
def _tail(normed, w, b):
    """forward_features' tail after the final LayerNorm (oracle/htsat_oracle.py forward_features): normed [B, 64, C] ->
    (y [B, 527, 32], framewise, clipwise, fine_grained_embedding, embedding)."""
    B, N, Cn = normed.shape
    x = normed.permute(0, 2, 1).reshape(B, Cn, 8, 8)
    x = x.reshape(B, Cn, 4, 2, 8).permute(0, 1, 3, 2, 4).reshape(B, Cn, 2, -1)
    fine = O.interpolate_repeat(torch.mean(x, dim=2).permute(0, 2, 1).contiguous(), 32)
    emb = torch.flatten(x, 2).mean(dim=-1)
    y = torch.flatten(F.conv2d(x, w, b, padding=(0, 1)), 2)
    fpx = O.interpolate_repeat(torch.sigmoid(y).permute(0, 2, 1).contiguous(), 32)
    return y, fpx, torch.sigmoid(y.mean(dim=-1)), fine, emb


def _tail_backward(model, precision, B=3, seed=0):
    """ard_tail_backward vs float64 autograd of _tail on the same fp32 normed tokens and output gradients."""
    clap, sd, _ = G.make_encoder(model)
    enc = clap.model.audio_branch
    h = enc._handle()
    NF = enc.num_features
    g = torch.Generator().manual_seed(seed)
    normed = torch.randn(B, 64, NF, generator=g)
    grads = [torch.randn(B, 1024, 527, generator=g), torch.randn(B, 527, generator=g), torch.randn(B, 1024, NF, generator=g),
             torch.randn(B, NF, generator=g)]
    nd = normed.double().requires_grad_(True)
    y, fpx, clip, fine, emb = _tail(nd, sd["tscam_conv.weight"].double(), sd["tscam_conv.bias"].double())
    sum((o * gg.double()).sum() for o, gg in zip((fpx, clip, fine, emb), grads)).backward()
    ydev = torch.zeros(B * 32, 528, device="cuda")
    ydev[:, :527] = y.detach().float().permute(0, 2, 1).reshape(B * 32, 527).cuda()
    gd = [t.cuda() for t in grads]
    out = torch.empty(B, 64, NF, device="cuda")
    L.check(L.load().ard_tail_backward(h, L.ptr(ydev), 528, L.ptr(gd[0]), L.ptr(gd[1]), L.ptr(gd[2]), L.ptr(gd[3]), B, precision, L.ptr(out),
                                       L.stream_ptr()))
    torch.cuda.synchronize()
    return G.rel(out, nd.grad)


@pytest.mark.parametrize("model", ["tiny", "base"])
def test_tail_backward_bf16(model):
    assert _tail_backward(model, 0) <= 5e-3


@pytest.mark.parametrize("model", ["tiny", "base"])
def test_tail_backward_fp32(model):
    assert _tail_backward(model, 1) <= 1e-5


# ---------------------------------------------------------------------------------------------------- op level: attention maps
ATTN_SHAPES = [(2, 64, 96, 4, 0), (2, 64, 96, 4, 4), (2, 32, 192, 8, 4), (3, 16, 384, 16, 4), (2, 8, 768, 32, 4), (2, 64, 128, 4, 4),
               (2, 16, 512, 16, 0)]   # test_window_attention_bwd's shapes


def _attention_pgrad_bwd(B, R, Cdim, nH, shift, fp32, scale=0.5, seed=0):
    """ard_window_attention(_f32)_bwd_pgrad vs float64 autograd of sum(out * dout) + scale * sum(P * pgrad) through the oracle's
    attention core (qkv / dout bf16-rounded for the bf16 kernel)."""
    g = torch.Generator().manual_seed(seed)
    hd = Cdim // nH
    T = R * R
    qkv = torch.randn(B * T, 3 * Cdim, generator=g)
    qkv[:, :Cdim] *= hd ** -0.5
    table = 0.5 * torch.randn(225, nH, generator=g)
    dout = torch.randn(B * T, Cdim, generator=g)
    nW = max(1, (R // 8) ** 2)
    pgrad = torch.randn(B * nW, nH, 64, 64, generator=g)
    if not fp32:
        qkv, dout = G.bf16r(qkv), G.bf16r(dout)
    qr = qkv.double().requires_grad_(True)
    out, attn = G._ref_window_attention(qr, table.double(), B, R, Cdim, nH, shift)
    ((out * dout.double()).sum() + scale * (attn * pgrad.double()).sum()).backward()
    dt = torch.float32 if fp32 else torch.bfloat16
    qd, dd, td, pd = qkv.to("cuda", dt), dout.to("cuda", dt), table.cuda(), pgrad.cuda()
    dq = torch.zeros(B * T, 3 * Cdim, device="cuda", dtype=dt)
    fn = L.load().ard_window_attention_f32_bwd_pgrad if fp32 else L.load().ard_window_attention_bwd_pgrad
    L.check(fn(L.ptr(qd), L.ptr(dd), L.ptr(pd), scale, L.ptr(dq), L.ptr(td), B, R, R, Cdim, nH, shift, L.stream_ptr()))
    torch.cuda.synchronize()
    got, ref = dq.float().cpu(), qr.grad
    return tuple(G.rel(got[:, i * Cdim:(i + 1) * Cdim], ref[:, i * Cdim:(i + 1) * Cdim]) for i in range(3))


@pytest.mark.parametrize("B,R,C,nH,shift", ATTN_SHAPES)
def test_window_attention_bwd_pgrad(B, R, C, nH, shift):
    m = _attention_pgrad_bwd(B, R, C, nH, shift, fp32=False)
    assert max(m) <= 5e-3, m


@pytest.mark.parametrize("B,R,C,nH,shift", ATTN_SHAPES)
def test_window_attention_f32_bwd_pgrad(B, R, C, nH, shift):
    m = _attention_pgrad_bwd(B, R, C, nH, shift, fp32=True)
    assert max(m) <= 1e-5, m


# ---------------------------------------------------------------------------------------------------- lambda gradients per key
def _functionals(enc, B, seed=11):
    """Fixed random linear functionals on framewise / fine-grained / each layers_residuals[l] / each layers_attention[l], and BCE
    targets for clipwise."""
    g = torch.Generator().manual_seed(seed)
    f = {"framewise_output": torch.randn(B, 1024, 527, generator=g) / 1024,
         "fine_grained_embedding": torch.randn(B, 1024, enc.num_features, generator=g) / 1024,
         "clip_target": (torch.rand(B, 527, generator=g) < 0.1).float()}
    for l in range(4):
        R = 64 >> l
        f[f"res{l}"] = torch.randn(B, enc.depths[l] * R * R, enc.embed_dim << l, generator=g) / (R * R)
        nW = max(1, (R // 8) ** 2)
        f[f"attn{l}"] = torch.randn(B * nW, enc.num_heads[l], 64, 64, generator=g) / nW
    return f


def _loss(out, key, f):
    """The loss of one key (or "all": their sum) on an output dict; functionals are moved to the output's device / dtype."""
    def fn(name):
        t = f[name]
        return t.to(device=out["embedding"].device, dtype=out["embedding"].dtype)
    if key == "all":
        return sum(_loss(out, k, f) for k in ("clipwise_output", "framewise_output", "fine_grained_embedding", 0, 1, 2, 3,
                                              "attn0", "attn1", "attn2", "attn3"))
    if key == "clipwise_output":
        return F.binary_cross_entropy(out["clipwise_output"], fn("clip_target"))
    if isinstance(key, int):
        return (out["layers_residuals"][key] * fn(f"res{key}")).sum()
    if key.startswith("attn"):
        return (out["layers_attention"][int(key[4:])] * fn(key)).sum()
    return (out[key] * fn(key)).sum()


KEYS = ("clipwise_output", "framewise_output", "fine_grained_embedding", 0, 1, 2, 3, "attn0", "attn1", "attn2", "attn3", "all")


def _oracle_grads(sd, model, ores, wave, keys, f, dtype):
    """d loss_k / d lambda_l through the oracle in `dtype` (one forward, one backward per key); None where lambda_l is unused."""
    lams = {l: lam.to(dtype).clone().requires_grad_(True) for l, (_, _, lam) in ores.items()}
    res = {l: (mu.to(dtype), comp.to(dtype), lams[l]) for l, (mu, comp, _) in ores.items()}
    out = O.htsat_forward({"waveform": wave.to(dtype)}, sd, W_CONFIGS[model], res)
    ls = sorted(lams)
    ref = {}
    for k in keys:
        loss = _loss(out, k, f)
        gs = torch.autograd.grad(loss, [lams[l] for l in ls], retain_graph=True, allow_unused=True) if loss.requires_grad else [None] * len(ls)
        ref[k] = dict(zip(ls, gs))
    return ref


W_CONFIGS = G.W.CONFIGS


def _lambda_grads(clap, wave, key, f, precision):
    """One training step of loss `key` through HTSAT_Swin_Transformer.forward: {layer: lambda.grad or None}."""
    enc = clap.model.audio_branch
    enc.train_precision = precision
    for r in clap._residuals.values():
        r.learnable.grad = None
    out = enc({"waveform": wave.cuda()})
    _loss(out, key, f).backward()
    torch.cuda.synchronize()
    return {l: (None if r.learnable.grad is None else r.learnable.grad.detach().cpu().clone()) for l, r in clap._residuals.items()}


def _per_key(model, layers, precision, keys=KEYS, B=2):
    clap, sd, ores = G.make_encoder(model, residual=tuple(layers))
    enc = clap.model.audio_branch
    wave = G.W.make_clips(B, seed=99)
    f = _functionals(enc, B)
    ref = _oracle_grads(sd, model, ores, wave, keys, f, torch.float64 if precision == "fp32" else torch.float32)
    got = {k: _lambda_grads(clap, wave, k, f, precision) for k in keys}
    return got, ref


def _errors(got, ref):
    m = {}
    for k in got:
        for l, gl in got[k].items():
            r = ref[k][l]
            if r is None or gl is None:
                m[(k, l)] = "none" if (r is None) == (gl is None) else ("got", gl is None, "ref", r is None)
            else:
                m[(k, l)] = G.rel(gl, r)
    return m


# Measured exceptions to the bf16 tier (B200). Every one of these cases meets the float64 oracle to 1e-4 at fp32 grade, so the
# schedule is exact and the excess is bf16 rounding:
# - lambda_0 for losses on layers_residuals[2] / [3] (all layers patched): 1.005e-2 / 1.006e-2, the bf16 dgrad operands through the
#   eight or more patched blocks between them (the tier of the reference's golden step is 1.2e-2 for the same reason, test_gpu_train.py);
# - losses on layers_attention: 1.0e-2 - 1.6e-2. The gradient of a map is taken through the softmax at the bf16 forward's
#   probabilities (bf16 q / k) with bf16 P / dS operands, and the maps themselves differ from the fp32 oracle's by that rounding.
def _bf16_tol(key):
    k, _ = key
    if k in (2, 3):
        return 1.2e-2
    if k in ("attn0", "attn1", "attn2", "attn3", "all"):
        return 3e-2
    return G.TOL_BF16


@pytest.mark.parametrize("precision,tol", [("bf16", G.TOL_BF16), ("fp32", G.TOL_FP32)])
@pytest.mark.parametrize("layers", [(0, 1, 2, 3), (1, 2)])
def test_lambda_grads_per_key_vs_oracle(precision, tol, layers):
    got, ref = _per_key("tiny", layers, precision)
    m = _errors(got, ref)
    tols = {k: (_bf16_tol(k) if precision == "bf16" else tol) for k in m}
    bad = {k: v for k, v in m.items() if not (v == "none" or (isinstance(v, float) and v <= tols[k]))}
    assert not bad, m


def test_base_fusion_clipwise_vs_oracle():
    """HTSAT-base with fusion, BCE on clipwise_output, fp32 grade against the float64 oracle."""
    clap, sd, ores = G.make_encoder("base", fusion=True, residual=True)
    enc = clap.model.audio_branch
    enc.train_precision = "fp32"
    B = 2
    wave = G.W.make_clips(B, seed=5)
    fb = torch.from_numpy(G.W.mel_filterbank(htk=True, slaney_norm=False)).float()
    win = torch.from_numpy(G.W.hann_periodic(1024)).float()
    mel = torch.stack([torch.stack([O.fusion_mel(w, fb, win)] * 4) for w in wave])
    f = _functionals(enc, B)
    for r in clap._residuals.values():
        r.learnable.grad = None
    out = enc({"mel_fusion": mel.cuda(), "longer": torch.zeros(B, 1)})
    _loss(out, "clipwise_output", f).backward()
    torch.cuda.synchronize()
    lams = {l: lam.double().clone().requires_grad_(True) for l, (_, _, lam) in ores.items()}
    res = {l: (mu.double(), comp.double(), lams[l]) for l, (mu, comp, _) in ores.items()}
    oout = O.htsat_forward({"mel_fusion": mel.double()}, sd, W_CONFIGS["base"], res, enable_fusion=True)
    _loss(oout, "clipwise_output", f).backward()
    m = {l: G.rel(r.learnable.grad, lams[l].grad) for l, r in clap._residuals.items()}
    assert max(m.values()) <= G.TOL_FP32, m


# ---------------------------------------------------------------------------------------------------- reachability, linearity
def test_residual_loss_reaches_only_lower_layers():
    """A loss on layers_residuals[1]: lambda_2 / lambda_3 get None (as reference autograd gives), lambda_0 / lambda_1 match."""
    got, ref = _per_key("tiny", (0, 1, 2, 3), "fp32", keys=(1,))
    assert got[1][2] is None and got[1][3] is None and ref[1][2] is None and ref[1][3] is None
    for l in (0, 1):
        assert G.rel(got[1][l], ref[1][l]) <= G.TOL_FP32, (l, G.rel(got[1][l], ref[1][l]))


@pytest.mark.parametrize("precision,tol", [("bf16", G.TOL_BF16), ("fp32", G.TOL_FP32)])
def test_attention_loss_reaches_lambda_of_its_own_layer(precision, tol):
    """Only layer 0 patched, a loss on layers_attention[0]: block 1's maps depend on block 0's lambda, so lambda_0 gets a non-zero
    gradient that matches the oracle (bf16: the attention-map bound of _bf16_tol)."""
    tol = _bf16_tol(("attn0", 0)) if precision == "bf16" else tol
    got, ref = _per_key("tiny", (0,), precision, keys=("attn0",))
    assert ref["attn0"][0] is not None and got["attn0"][0] is not None and got["attn0"][0].abs().max() > 0
    assert G.rel(got["attn0"][0], ref["attn0"][0]) <= tol, G.rel(got["attn0"][0], ref["attn0"][0])


def test_sum_of_keys_is_linear_fp32():
    """The gradient of the summed loss is the sum of the per-key gradients. To 2e-5, not to fp32 rounding: every fp32-grade dgrad
    splits its fp32 operand into bf16 hi + lo (16 significant bits, 2^-17 relative), and the split of a sum is not the sum of the
    splits (measured 9.3e-6 on lambda_0, B200)."""
    clap, _, _ = G.make_encoder("tiny", residual=True)
    wave = G.W.make_clips(2, seed=99)
    f = _functionals(clap.model.audio_branch, 2)
    keys = ("clipwise_output", "framewise_output", "fine_grained_embedding", 0, 1, 2, 3, "attn0", "attn1", "attn2", "attn3")
    per = [_lambda_grads(clap, wave, k, f, "fp32") for k in keys]
    tot = _lambda_grads(clap, wave, "all", f, "fp32")
    for l, t in tot.items():
        s = sum(p[l] for p in per if p[l] is not None)
        assert G.rel(t, s) <= 2e-5, (l, G.rel(t, s))


# ---------------------------------------------------------------------------------------------------- today's losses unchanged
def test_audio_embed_loss_unchanged_by_want_dict():
    """A loss on audio_embed alone: the same lambda gradient and the same backward launches whether or not the forward also
    computed the tail and the captures. (The lambda reductions use float atomics, so two identical steps may differ in the last
    bits: the comparison is against that spread.)"""
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(2, seed=1234).cuda()
    lib = L.load()

    def step(want_dict):
        for r in clap._residuals.values():
            r.learnable.grad = None
        out = enc.encode(waveform=wave, want_audio_embed=True, want_dict=want_dict)
        torch.cuda.synchronize()
        lib.ard_launch_counter_reset()
        out["audio_embed"].sum().backward()
        torch.cuda.synchronize()
        n = lib.ard_launch_counter_read()
        return torch.cat([r.learnable.grad.detach().cpu().flatten() for _, r in sorted(clap._residuals.items())]), n

    g0, n0 = step(False)
    g0b, _ = step(False)
    g1, n1 = step(True)
    spread = G.rel(g0b, g0)
    assert n0 == n1, (n0, n1)
    assert torch.equal(g1, g0) or G.rel(g1, g0) <= max(2 * spread, 1e-6), (G.rel(g1, g0), spread)


# ---------------------------------------------------------------------------------------------------- C ABI error paths
def test_tail_gradient_needs_saved_tail():
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    wave = G.W.make_clips(1, seed=3).cuda()
    lib = L.load()
    dl = {l: torch.zeros(int(r.learnable.shape[0]), device="cuda") for l, r in clap._residuals.items()}
    gc = torch.zeros(1, 527, device="cuda")
    ga = torch.zeros(64, 4, 64, 64, device="cuda")   # layers_attention[0] of one clip: 64 windows, 4 heads

    def call(gen, **grads):
        a = L.ArdBackwardArgs()
        a.B, a.generation = 1, gen
        for l, t in dl.items():
            a.grad_lambda[l] = t.data_ptr()
        o = L.ArdOutputGrads()
        for k, v in grads.items():
            if k == "attn0":
                o.grad_layers_attention[0] = v.data_ptr()
            else:
                setattr(o, k, v.data_ptr())
        return lib.ard_encoder_backward_outputs(enc._hb.h, C.byref(a), C.byref(o), L.stream_ptr())

    with torch.no_grad():
        gen = enc.encode(waveform=wave, save_for_backward=True)["_tape_generation"]
    assert call(gen, grad_clipwise_output=gc) == L.ARD_ERR_STATE
    assert call(gen) == L.ARD_ERR_SHAPE                                   # no output gradient at all
    with torch.no_grad():
        gen = enc.encode(waveform=wave, save_for_backward=True, want_dict=True)["_tape_generation"]
    assert call(gen, attn0=ga) == 0
    assert call(gen, grad_clipwise_output=gc) == 0
    torch.cuda.synchronize()
