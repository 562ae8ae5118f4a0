"""Host-side mirror of the reference's HTSAT module API, backed by libard_b200.so.

Mirrors CLAP/src/laion_clap/clap_module/htsat.py: same class names, constructor arguments, module tree and therefore
the same state_dict keys (`layers.{l}.blocks.{b}.attn.qkv.weight`, `bn0.running_mean`, `logmel_extractor.melW`, ...), the
same `forward(x: dict, mixup_lambda=None, infer_mode=False, device=None) -> output_dict` with the six keys of
htsat.py:825-832, and `model.layers[l].blocks[b]` stays addressable (src/residual.py:194,204-205 relies on it).
The modules only HOLD parameters; all arithmetic runs in hand-written sm_100a kernels through the C ABI. Eval-mode
semantics only: the reference forces `.eval()` on every call path that reaches the encoder (hook.py:173, SURVEY Q5).
"""
import copy
import ctypes as C
import weakref

import torch
import torch.nn as nn

from . import lib as L

WINDOW = 8


class _HandleBox:
    """Owns the opaque ard_handle*. Never deep-copied: a copy of the encoder lazily creates its own handle."""

    def __init__(self):
        self.h = None
        self.sig = None         # weight signature last pushed
        self.res_sig = {}       # (layer, block) -> signature of the injected ResiDual

    def __deepcopy__(self, memo):
        return _HandleBox()

    def __del__(self):
        try:
            if self.h is not None:
                L.load().ard_destroy(self.h)
        except Exception:
            pass


class _Holder(nn.Module):
    """Parameter container whose only job is to reproduce a reference module's parameter names."""

    def forward(self, *a, **k):
        raise RuntimeError("parameter holder: arithmetic runs in libard_b200.so")


class _ConvW(_Holder):
    def __init__(self, shape, bias=False):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(*shape), requires_grad=False)
        if bias:
            self.bias = nn.Parameter(torch.zeros(shape[0]), requires_grad=False)


class _STFT(_Holder):
    def __init__(self, n_fft):
        super().__init__()
        self.conv_real = _ConvW((n_fft // 2 + 1, 1, n_fft))
        self.conv_imag = _ConvW((n_fft // 2 + 1, 1, n_fft))


class Spectrogram(_Holder):          # torchlibrosa.stft.Spectrogram as built at htsat.py:681-683
    def __init__(self, n_fft):
        super().__init__()
        self.stft = _STFT(n_fft)


class LogmelFilterBank(_Holder):     # torchlibrosa.stft.LogmelFilterBank, htsat.py:685-687
    def __init__(self, n_fft, n_mels):
        super().__init__()
        self.melW = nn.Parameter(torch.zeros(n_fft // 2 + 1, n_mels), requires_grad=False)


class Mlp(_Holder):                  # htsat.py:146-164
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class WindowAttention(_Holder):      # htsat.py:278-360
    def __init__(self, dim, window_size, num_heads):
        super().__init__()
        self.dim, self.window_size, self.num_heads = dim, (window_size, window_size), num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * window_size - 1) ** 2, num_heads))
        coords = torch.stack(torch.meshgrid([torch.arange(window_size), torch.arange(window_size)], indexing="ij"))
        cf = torch.flatten(coords, 1)
        rel = (cf[:, :, None] - cf[:, None, :]).permute(1, 2, 0).contiguous()
        rel[:, :, 0] += window_size - 1
        rel[:, :, 1] += window_size - 1
        rel[:, :, 0] *= 2 * window_size - 1
        self.register_buffer("relative_position_index", rel.sum(-1))
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)


class SwinTransformerBlock(nn.Module):
    """htsat.py:363-487. forward(x[B, H*W, C]) -> (x, attn[B*nW, nH, 64, 64], residual_x[B, H*W, C])."""

    def __init__(self, dim, input_resolution, num_heads, window_size=8, shift_size=0, mlp_ratio=4.0):
        super().__init__()
        self.dim, self.input_resolution, self.num_heads = dim, input_resolution, num_heads
        self.window_size, self.shift_size, self.mlp_ratio = window_size, shift_size, mlp_ratio
        if min(input_resolution) <= window_size:   # htsat.py:393-396
            self.shift_size = 0
            self.window_size = min(input_resolution)
        assert 0 <= self.shift_size < self.window_size, "shift_size must in 0-window_size"
        self.norm1 = nn.LayerNorm(dim)
        self.attn = WindowAttention(dim, self.window_size, num_heads)
        self.drop_path = nn.Identity()
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))
        if self.shift_size > 0:                    # htsat.py:414-435 (kept as a buffer for state_dict parity)
            H, W = input_resolution
            img_mask = torch.zeros((1, H, W, 1))
            cnt = 0
            for h in (slice(0, -self.window_size), slice(-self.window_size, -self.shift_size), slice(-self.shift_size, None)):
                for w in (slice(0, -self.window_size), slice(-self.window_size, -self.shift_size), slice(-self.shift_size, None)):
                    img_mask[:, h, w, :] = cnt
                    cnt += 1
            ws = self.window_size
            mw = img_mask.view(1, H // ws, ws, W // ws, ws, 1).permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, ws * ws)
            am = mw.unsqueeze(1) - mw.unsqueeze(2)
            attn_mask = am.masked_fill(am != 0, float(-100.0)).masked_fill(am == 0, float(0.0))
        else:
            attn_mask = None
        self.register_buffer("attn_mask", attn_mask)
        object.__setattr__(self, "_enc_ref", None)     # weakref to the owning encoder (not a submodule)
        object.__setattr__(self, "_residual", None)    # ResiDual injected by patch_block_with_residual (not registered, SURVEY Q4)
        self._index = (0, 0)

    def _encoder(self):
        enc = self._enc_ref() if self._enc_ref is not None else None
        if enc is None:
            raise RuntimeError("SwinTransformerBlock is not attached to an HTSAT_Swin_Transformer")
        return enc

    def forward(self, x):
        return self._encoder()._block_forward(self, x)

    def extra_repr(self):
        return (f"dim={self.dim}, input_resolution={self.input_resolution}, num_heads={self.num_heads}, "
                f"window_size={self.window_size}, shift_size={self.shift_size}, mlp_ratio={self.mlp_ratio}")


class PatchMerging(_Holder):         # htsat.py:490-529
    def __init__(self, input_resolution, dim):
        super().__init__()
        self.input_resolution, self.dim = input_resolution, dim
        self.reduction = nn.Linear(4 * dim, 2 * dim, bias=False)
        self.norm = nn.LayerNorm(4 * dim)


class BasicLayer(nn.Module):         # htsat.py:532-600
    def __init__(self, dim, input_resolution, depth, num_heads, window_size, downsample):
        super().__init__()
        self.dim, self.input_resolution, self.depth = dim, input_resolution, depth
        self.blocks = nn.ModuleList([
            SwinTransformerBlock(dim, input_resolution, num_heads, window_size, 0 if i % 2 == 0 else window_size // 2)
            for i in range(depth)])
        self.downsample = PatchMerging(input_resolution, dim) if downsample else None


class PatchEmbed(_Holder):           # htsat.py:71-144
    def __init__(self, img_size, patch_size, in_chans, embed_dim, enable_fusion, fusion_type):
        super().__init__()
        self.img_size, self.patch_size = (img_size, img_size), (patch_size, patch_size)
        self.grid_size = (img_size // patch_size, img_size // patch_size)
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.norm = nn.LayerNorm(embed_dim)
        # The aff_2d fusion branch (mel_conv2d + AFF, htsat.py:104-134) only runs for clips > 10 s, which the reference
        # cannot reach (data.py:467 crashes, SURVEY Q9/Q14); its 23,616 parameters are not instantiated here.


class HTSAT_Swin_Transformer(nn.Module):
    """htsat.py:596-994 (eval-mode routes). All arithmetic runs in libard_b200.so."""

    def __init__(self, spec_size=256, patch_size=4, patch_stride=(4, 4), in_chans=1, num_classes=527, embed_dim=96,
                 depths=(2, 2, 6, 2), num_heads=(4, 8, 16, 32), window_size=8, mlp_ratio=4.0, config=None,
                 enable_fusion=False, fusion_type="None", joint_dim=512, **kwargs):
        super().__init__()
        self.config = config
        self.spec_size, self.patch_size, self.patch_stride = spec_size, patch_size, tuple(patch_stride)
        self.window_size, self.embed_dim, self.depths, self.num_heads = window_size, embed_dim, list(depths), list(num_heads)
        self.in_chans, self.num_classes, self.mlp_ratio = in_chans, num_classes, mlp_ratio
        self.num_layers = len(self.depths)
        self.num_features = int(embed_dim * 2 ** (self.num_layers - 1))
        self.enable_fusion, self.fusion_type = enable_fusion, fusion_type
        self.joint_dim = joint_dim
        mel_bins = getattr(config, "mel_bins", 64) if config is not None else 64
        n_fft = getattr(config, "window_size", 1024) if config is not None else 1024
        if spec_size != 256 or patch_size != 4 or window_size != 8 or mel_bins != 64 or n_fft != 1024 or len(self.depths) != 4:
            raise RuntimeError("Import Model not found, or the audio cfg parameters are not enough.")   # htsat.py:1044-1045
        self.freq_ratio = spec_size // mel_bins
        self.spectrogram_extractor = Spectrogram(n_fft)
        self.logmel_extractor = LogmelFilterBank(n_fft, mel_bins)
        self.bn0 = nn.BatchNorm2d(mel_bins)
        self.patch_embed = PatchEmbed(spec_size, patch_size, in_chans, embed_dim, enable_fusion, fusion_type)
        res = self.patch_embed.grid_size
        self.patches_resolution = res
        self.layers = nn.ModuleList([
            BasicLayer(int(embed_dim * 2 ** i), (res[0] // 2 ** i, res[1] // 2 ** i), self.depths[i], self.num_heads[i],
                       window_size, downsample=i < self.num_layers - 1) for i in range(self.num_layers)])
        self.norm = nn.LayerNorm(self.num_features)
        SF = spec_size // (2 ** (self.num_layers - 1)) // self.patch_stride[0] // self.freq_ratio
        self.tscam_conv = nn.Conv2d(self.num_features, num_classes, kernel_size=(SF, 3), padding=(0, 1))
        self.head = nn.Linear(num_classes, num_classes)   # present (unused) in the reference too, htsat.py:748
        # CLAP-level projection (model.py:539-543) rides on the same handle; set by CLAP.__init__
        object.__setattr__(self, "_projection", None)
        self.train_precision = "bf16"
        self._hb = _HandleBox()
        self._relink()
        for p in self.parameters():
            p.requires_grad = False
        self.eval()

    # ------------------------------------------------------------------ plumbing
    def _relink(self):
        ref = weakref.ref(self)
        for l, layer in enumerate(self.layers):
            for b, blk in enumerate(layer.blocks):
                object.__setattr__(blk, "_enc_ref", ref)
                blk._index = (l, b)

    def __deepcopy__(self, memo):    # setup_residual_htsat deep-copies the encoder (src/residual.py:186)
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = copy.deepcopy(v, memo)
        new._relink()
        return new

    @property
    def train_precision(self):
        """Precision of the training step (the autograd route into the ResiDual lambdas): "bf16" (default, the tensor-core
        path) or "fp32" (3-term split-bf16 GEMMs forward and backward, fp32 attention / LayerNorm / GELU backward; the lambda
        gradients then match the reference's fp32 loss.backward() to rel. err <= 1e-4)."""
        return self.__dict__.get("_train_precision", "bf16")

    @train_precision.setter
    def train_precision(self, value):
        if value not in ("bf16", "fp32"):
            raise ValueError(f"train_precision must be 'bf16' or 'fp32' (got {value!r})")
        object.__setattr__(self, "_train_precision", value)

    def _device(self):
        return self.norm.weight.device

    def _audio_keys(self):
        skip = ("relative_position_index", "attn_mask", "num_batches_tracked")
        for k, v in self.state_dict().items():
            if k.endswith(skip) or k.startswith("head."):
                continue
            if self.enable_fusion and (k.startswith("spectrogram_extractor") or k.startswith("logmel_extractor")):
                continue
            yield k, v

    def _signature(self):
        sig = [(k, v.data_ptr(), v._version) for k, v in self._audio_keys()]
        if self._projection is not None:
            sig += [(k, v.data_ptr(), v._version) for k, v in self._projection.state_dict().items()]
        return tuple(sig)

    def _handle(self):
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("audio_residual_b200 runs on CUDA (sm_100a) only: move the model to a GPU; there is no CPU fallback")
        lib = L.load()
        hb = self._hb
        with torch.cuda.device(dev):
            if hb.h is None:
                cfg = L.ArdConfig(self.embed_dim, (C.c_int * 4)(*self.depths), (C.c_int * 4)(*self.num_heads), self.joint_dim,
                                  int(bool(self.enable_fusion)))
                h = C.c_void_p()
                L.check(lib.ard_create(C.byref(cfg), C.byref(h)), RuntimeError)
                hb.h, hb.sig, hb.res_sig = h, None, {}
            sig = self._signature()
            if sig != hb.sig:
                items = list(self._audio_keys())
                if self._projection is not None:
                    items += [("audio_projection." + k, v) for k, v in self._projection.state_dict().items()]
                if self.enable_fusion:
                    # constants of the fusion featuriser get_mel (data.py:365-378): torchaudio's htk filterbank (norm=None)
                    # and torch.hann_window(1024) (periodic); they are not checkpoint tensors
                    from . import weights as W
                    items += [("fusion_featuriser.melW", torch.from_numpy(W.mel_filterbank(htk=True, slaney_norm=False))),
                              ("fusion_featuriser.window", torch.from_numpy(W.hann_periodic(1024)))]
                for k, v in items:
                    t = v.detach().to("cpu", torch.float32).contiguous()
                    L.check(lib.ard_set_weight(hb.h, k.encode(), L.ptr(t), t.numel()))
                L.check(lib.ard_finalize_weights(hb.h, L.stream_ptr()))
                hb.sig = sig
                hb.res_sig = {}
            self._sync_residuals(lib)
        return hb.h

    def _sync_residuals(self, lib):
        hb, dev = self._hb, self._device()
        for l, layer in enumerate(self.layers):
            stale = []   # patched blocks whose folded projection must be re-derived: (block index, ResiDual, basis signature, lambda signature)
            for b, blk in enumerate(layer.blocks):
                res = blk._residual
                key = (l, b)
                if res is None:
                    if key in hb.res_sig:
                        L.check(lib.ard_clear_block_residual(hb.h, l, b))
                        del hb.res_sig[key]
                    continue
                bsig = (id(res), res.basis.data_ptr(), res.basis._version, res.mean.data_ptr(), res.mean._version)
                lsig = (res.learnable.data_ptr(), res.learnable._version)
                old = hb.res_sig.get(key)
                if old is None or old[0] != bsig:
                    basis = res.basis.detach().to("cpu", torch.float32).contiguous()
                    mean = res.mean.detach().to("cpu", torch.float32).contiguous()
                    L.check(lib.ard_set_block_residual(hb.h, l, b, L.ptr(mean), L.ptr(basis), basis.shape[0], basis.shape[1]))
                    old = None
                if old is None or old[1] != lsig:
                    stale.append((b, res, bsig, lsig))
            if not stale:
                continue
            patched = [blk._residual for blk in layer.blocks if blk._residual is not None]
            shared = len(stale) == len(patched) and len(patched) > 1 and all(r is patched[0] for r in patched)
            if shared:
                # one ResiDual per layer shared by its blocks (src/residual.py:170-186): M once, the blocks' folds batched
                res = patched[0]
                lam = res.learnable.detach().to(dev, torch.float32).contiguous()   # reference re-copies per call (Q4)
                L.check(lib.ard_set_layer_lambda(hb.h, l, L.ptr(lam), L.stream_ptr()))
                res._lam_dev = lam
            for b, res, bsig, lsig in stale:
                if not shared:
                    lam = res.learnable.detach().to(dev, torch.float32).contiguous()
                    L.check(lib.ard_set_block_lambda(hb.h, l, b, L.ptr(lam), L.stream_ptr()))
                    res._lam_dev = lam
                hb.res_sig[(l, b)] = (bsig, lsig)

    # ------------------------------------------------------------------ compute
    def _block_forward(self, blk, x):
        l, b = blk._index
        H, W = blk.input_resolution
        B, Ltok, Cc = x.shape
        if Ltok != H * W or Cc != blk.dim:
            raise ValueError(f"input feature has wrong size: got {tuple(x.shape)}, block expects [B, {H * W}, {blk.dim}]")
        h = self._handle()
        lib = L.load()
        x = x.detach().to(self._device(), torch.float32).contiguous()
        nW = (H // blk.window_size) * (W // blk.window_size)
        out = torch.empty_like(x)
        attn = torch.empty((B * nW, blk.num_heads, 64, 64), device=x.device, dtype=torch.float32)
        res = torch.empty_like(x)
        with torch.cuda.device(x.device):
            L.check(lib.ard_block_forward(h, l, b, L.ptr(x), B, L.ptr(out), L.ptr(attn), L.ptr(res), L.stream_ptr()))
        return out, attn, res

    def _lambda_params(self):
        """Per layer: the ResiDual `learnable` parameter shared by that layer's patched blocks (src/residual.py:186-197), or None."""
        out = []
        for layer in self.layers:
            res = {id(b._residual): b._residual for b in layer.blocks if b._residual is not None}
            if len(res) > 1:
                raise NotImplementedError("blocks of one layer must share a single ResiDual module (setup_residual_htsat does)")
            out.append(next(iter(res.values())).learnable if res else None)
        return out

    def encode(self, waveform=None, mel_fusion=None, quantize=False, want_dict=False, want_audio_embed=False,
               want_capture=True, save_for_backward=False, want_head_outputs=False, precision=None):
        """Single entry to ard_encoder_forward. Returns a dict of freshly allocated CUDA tensors.
        With grad enabled and trainable ResiDual lambdas, every output the reference can differentiate w.r.t. the lambdas comes back
        attached to the autograd graph: `embedding`, `audio_embed`, `framewise_output`, `clipwise_output`, `fine_grained_embedding`
        and each tensor of `layers_residuals` and `layers_attention` (backward = ard_encoder_backward_outputs, filling
        `learnable.grad` as loss.backward() does in src/training.py:30-32; a lambda no used output depends on gets no gradient).
        `head_outputs` is not a reference output and is never differentiable.
        want_head_outputs: also return `head_outputs`, per layer [depth, B*nW, nH, 64, hd]: every block's per-head `attn @ v`
        (htsat.py:354). precision: "bf16" (default) or "fp32" (3-term split-bf16 GEMMs + fp32 attention, rel. err <= 1e-4);
        None takes the encoder's `precision` attribute. The autograd route runs at the encoder's `train_precision` instead;
        an encoder set to precision="fp32" trains only with train_precision="fp32" too (never silently in bf16).
        save_for_backward=True with precision="fp32" saves an fp32-grade forward for an fp32-grade backward."""
        precision = precision or getattr(self, "precision", "bf16")
        if precision not in ("bf16", "fp32"):
            raise ValueError(f"precision must be 'bf16' or 'fp32' (got {precision!r})")
        if not save_for_backward and torch.is_grad_enabled():
            lams = self._lambda_params()
            if any(p is not None and p.requires_grad for p in lams):
                if precision != "bf16" and self.train_precision != "fp32":
                    raise NotImplementedError(f"precision={precision!r} with train_precision={self.train_precision!r}: the training step "
                                              "runs at train_precision; set train_precision='fp32' to train at fp32 grade")
                return _encode_with_grad(self, lams, waveform, mel_fusion, quantize, want_dict, want_audio_embed, want_capture,
                                         self.train_precision)
        h = self._handle()
        lib = L.load()
        dev = self._device()
        src = mel_fusion if self.enable_fusion else waveform
        if src is None:
            raise ValueError("fusion model expects 'mel_fusion', non-fusion model expects 'waveform'")
        src = src.detach().to(dev, torch.float32).contiguous()
        B = src.shape[0]
        if self.enable_fusion:
            if src.dim() != 4 or src.shape[1] != 4 or src.shape[2] > 1024 or src.shape[3] != 64:
                raise AssertionError("the wav size should less than or equal to the swin input size")   # htsat.py:852
            if src.shape[2] != 1001:
                raise NotImplementedError("mel_fusion must have 1001 frames (10 s clips)")
        elif src.dim() != 2 or src.shape[1] != 480000:
            raise AssertionError(f"waveform must be [B, 480000] (got {tuple(src.shape)}): pad/crop with get_audio_features first")
        f32 = dict(device=dev, dtype=torch.float32)
        out = {"embedding": torch.empty((B, self.num_features), **f32)}
        a = L.ArdForwardArgs()
        a.B, a.quantize = B, int(bool(quantize))
        a.save_for_backward = int(bool(save_for_backward))
        a.precision = 1 if precision == "fp32" else 0
        if self.enable_fusion:
            a.mel_fusion = src.data_ptr()
        else:
            a.waveform = src.data_ptr()
        a.embedding = out["embedding"].data_ptr()
        if want_audio_embed:
            out["audio_embed"] = torch.empty((B, self.joint_dim), **f32)
            a.audio_embed = out["audio_embed"].data_ptr()
        if want_dict:
            out["framewise_output"] = torch.empty((B, 1024, self.num_classes), **f32)
            out["clipwise_output"] = torch.empty((B, self.num_classes), **f32)
            out["fine_grained_embedding"] = torch.empty((B, 1024, self.num_features), **f32)
            a.framewise_output = out["framewise_output"].data_ptr()
            a.clipwise_output = out["clipwise_output"].data_ptr()
            a.fine_grained_embedding = out["fine_grained_embedding"].data_ptr()
            if want_capture:
                attns, ress = [], []
                for l in range(self.num_layers):
                    Cl, R = self.embed_dim << l, 64 >> l
                    nW = max(1, (R // 8) * (R // 8))
                    attns.append(torch.empty((B * nW, self.num_heads[l], 64, 64), **f32))
                    ress.append(torch.empty((B, self.depths[l] * R * R, Cl), **f32))
                    a.layers_attention[l] = attns[l].data_ptr()
                    a.layers_residuals[l] = ress[l].data_ptr()
                out["layers_attention"], out["layers_residuals"] = attns, ress
        if want_head_outputs:
            taps = []
            for l in range(self.num_layers):
                Cl, R = self.embed_dim << l, 64 >> l
                nW = max(1, (R // 8) * (R // 8))
                taps.append(torch.empty((self.depths[l], B * nW, self.num_heads[l], 64, Cl // self.num_heads[l]), **f32))
                a.head_outputs[l] = taps[l].data_ptr()
            out["head_outputs"] = taps
        with torch.cuda.device(dev):
            L.check(lib.ard_encoder_forward(h, C.byref(a), L.stream_ptr()))
            if save_for_backward:
                out["_tape_generation"] = int(lib.ard_tape_generation(h))
        out["_keepalive"] = src
        return out

    def fusion_mel(self, wave, quantize=False):
        """Batched get_mel + 4x stack (data.py:363-399, :497-501) on device: wave [B, 480000] -> mel_fusion [B, 4, 1001, 64]."""
        h = self._handle()
        wave = wave.detach().to(self._device(), torch.float32).contiguous()
        B, n = wave.shape
        out = torch.empty((B, 4, n // 480 + 1, 64), device=wave.device, dtype=torch.float32)
        with torch.cuda.device(wave.device):
            L.check(L.load().ard_fusion_mel(h, L.ptr(wave), B, n, int(bool(quantize)), L.ptr(out), L.stream_ptr()))
        return out

    def forward(self, x, mixup_lambda=None, infer_mode=False, device=None):
        """htsat.py:881-994. x: {"waveform": [B,480000]} or, with fusion, {"mel_fusion": [B,4,1001,64], "longer": [B,1]}."""
        if self.training:
            raise NotImplementedError("train-mode HTSAT (SpecAugment/mixup/DropPath) is outside the ResiDual path: the "
                                      "reference always runs the encoder in eval mode (hook.py:173)")
        if self.enable_fusion:
            if "longer" in x and bool(torch.as_tensor(x["longer"]).sum() > 0):
                raise NotImplementedError("clips longer than 10 s are unreachable in the reference (data.py:467)")
            out = self.encode(mel_fusion=x["mel_fusion"], want_dict=True)
        else:
            out = self.encode(waveform=x["waveform"], want_dict=True)
        return {k: out[k] for k in ("framewise_output", "clipwise_output", "fine_grained_embedding", "embedding",
                                    "layers_attention", "layers_residuals")}

    def last_launch_count(self):
        return L.load().ard_last_launch_count(self._hb.h) if self._hb.h is not None else 0


_TAIL_KEYS = ("framewise_output", "clipwise_output", "fine_grained_embedding")


class _EncodeFn(torch.autograd.Function):
    """autograd node around ard_encoder_forward(save_for_backward=1) / ard_encoder_backward_outputs. Inputs: the per-layer lambda
    parameters (only to receive gradients; their values reach the library through _sync_residuals). Outputs: every tensor of the
    forward's output dict that the reference can differentiate w.r.t. ResiDual.learnable (htsat.py:797-832): `embedding`,
    `audio_embed`, the tail keys and the per-layer captures. Unused outputs get no gradient tensor (set_materialize_grads(False))
    and reach the library as NULL."""

    @staticmethod
    def forward(ctx, enc, kw, holder, *lams):
        ctx.set_materialize_grads(False)
        out = enc.encode(save_for_backward=True, **kw)
        holder.update(out)
        ctx.enc, ctx.B = enc, out["embedding"].shape[0]
        ctx.generation = out["_tape_generation"]   # the handle keeps ONE tape: a later training forward invalidates this node
        ctx.layers = [i for i, p in enumerate(enc._lambda_params()) if p is not None]
        ctx.ks = [p.shape[0] for p in enc._lambda_params() if p is not None]
        ctx.devs = [p.device for p in enc._lambda_params() if p is not None]
        # lambda_l acts from the first patched block of layer l on; a layer's attention maps are those of blocks after it
        ctx.attn_reach = {l: next(b for b, blk in enumerate(enc.layers[l].blocks) if blk._residual is not None) < enc.depths[l] - 1
                          for l in ctx.layers}
        ctx.keys = _output_keys(out, enc.num_layers)
        return tuple(out[k] if l is None else out[k][l] for k, l in ctx.keys)

    @staticmethod
    def backward(ctx, *grads):
        enc = ctx.enc
        dev = enc._device()
        lib = L.load()
        a = L.ArdBackwardArgs()
        a.B = ctx.B
        a.generation = ctx.generation
        o = L.ArdOutputGrads()
        keep = []
        # what the given gradients reach: everything (a head / tail key), the lambdas of layers <= top_res (residuals: the
        # patched blocks' own r), and those of layers < top_attn, or == top_attn with a block after the first patched one
        head, top_res, top_attn = False, -1, -1
        for (k, l), g in zip(ctx.keys, grads):
            if g is None:
                continue
            g = g.detach().to(dev, torch.float32).contiguous()
            keep.append(g)
            if k == "layers_residuals":
                o.grad_layers_residuals[l] = g.data_ptr()
                top_res = max(top_res, l)
                continue
            if k == "layers_attention":
                o.grad_layers_attention[l] = g.data_ptr()
                top_attn = max(top_attn, l)
                continue
            head = True
            if k == "embedding":
                a.grad_embedding = g.data_ptr()
            elif k == "audio_embed":
                a.grad_audio_embed = g.data_ptr()
            else:
                setattr(o, "grad_" + k, g.data_ptr())
        # lambda_l reaches every output from its first patched block on: the head and tail, and the residuals of layers >= l
        reached = [head or l <= top_res or l < top_attn or (l == top_attn and ctx.attn_reach[l]) for l in ctx.layers]
        outs = {}
        for l, k in zip(ctx.layers, ctx.ks):
            outs[l] = torch.empty(k, device=dev, dtype=torch.float32)
            a.grad_lambda[l] = outs[l].data_ptr()
        if any(reached):
            with torch.cuda.device(dev):
                L.check(lib.ard_encoder_backward_outputs(enc._hb.h, C.byref(a), C.byref(o), L.stream_ptr()))
        return (None, None, None) + tuple(outs[l].to(d) if r else None for l, d, r in zip(ctx.layers, ctx.devs, reached))


def _encode_with_grad(enc, lams, waveform, mel_fusion, quantize, want_dict, want_audio_embed, want_capture, precision):
    kw = dict(waveform=waveform, mel_fusion=mel_fusion, quantize=quantize, want_dict=want_dict, want_audio_embed=want_audio_embed,
              want_capture=want_capture, precision=precision)
    holder = {}
    live = [p for p in lams if p is not None]
    res = _EncodeFn.apply(enc, kw, holder, *live)
    out = {k: list(v) if isinstance(v, list) else v for k, v in holder.items()}
    for i, (k, l) in enumerate(_output_keys(holder, enc.num_layers)):
        if l is None:
            out[k] = res[i]
        else:
            out[k][l] = res[i]
    return out


def _output_keys(out, num_layers):
    """The differentiable outputs of _EncodeFn in order (the same list its forward builds)."""
    keys = [("embedding", None)] + [(k, None) for k in ("audio_embed",) + _TAIL_KEYS if k in out]
    if "layers_residuals" in out:
        keys += [(k, l) for k in ("layers_residuals", "layers_attention") for l in range(num_layers)]
    return keys


def create_htsat_model(audio_cfg, enable_fusion=False, fusion_type="None"):
    """htsat.py:996-1045."""
    name = audio_cfg.model_name if hasattr(audio_cfg, "model_name") else audio_cfg["model_name"]
    classes = audio_cfg.class_num if hasattr(audio_cfg, "class_num") else audio_cfg.get("class_num", 527)
    try:
        assert name in ["tiny", "base"], "model name for HTS-AT is wrong!"
        dims = {"tiny": (96, (2, 2, 6, 2)), "base": (128, (2, 2, 12, 2))}[name]
        return HTSAT_Swin_Transformer(spec_size=256, patch_size=4, patch_stride=(4, 4), num_classes=classes, embed_dim=dims[0],
                                      depths=dims[1], num_heads=(4, 8, 16, 32), window_size=8, config=None,
                                      enable_fusion=enable_fusion, fusion_type=fusion_type)
    except Exception:
        raise RuntimeError(f"Import Model for {name} not found, or the audio cfg parameters are not enough.")
