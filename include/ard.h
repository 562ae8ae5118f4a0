/*
 * ard.h — C ABI of libard_b200.so: the B200 (sm_100a) implementation of Audio-ResiDual's HTSAT + ResiDual hot path.
 *
 * Drop-in boundary. The reference (arianna011/Audio-ResiDual) is pure Python/PyTorch and has NO foreign-function
 * interface of its own, so each entry point below names the reference Python interface it replaces (paths relative to
 * the reference root). The reference-side binding is a ctypes stub; see INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer owned by the caller (PyTorch
 *     allocator on the reference side) and borrowed for the duration of the call; outputs are written in place.
 *   - every function returns 0 on success or a negative ARD_ERR_* code; ard_last_error() returns the message of the
 *     last failure on the calling thread. No exceptions, no exit(). The Python shim maps codes back to the exception
 *     types the reference raises (ValueError / AssertionError / RuntimeError / NotImplementedError).
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream); calls are asynchronous.
 *   - one ard_handle per device; a handle is not thread-safe, distinct handles are independent.
 */
#ifndef ARD_H_
#define ARD_H_

#ifdef __cplusplus
extern "C" {
#endif

#define ARD_OK 0
#define ARD_ERR_SHAPE (-1)    /* bad shape / index  -> ValueError or AssertionError (htsat.py:115,137,511; src/residual.py:194) */
#define ARD_ERR_DTYPE (-2)
#define ARD_ERR_CUDA (-3)     /* CUDA runtime/driver failure -> RuntimeError */
#define ARD_ERR_STATE (-4)    /* weights missing / not finalised -> RuntimeError */
#define ARD_ERR_KEY (-5)      /* unknown state_dict key -> KeyError */
#define ARD_ERR_NOTIMPL (-6)  /* -> NotImplementedError (data.py:462-464,494-496) */

#define ARD_ACT_NONE 0
#define ARD_ACT_GELU 1  /* exact-erf GELU, htsat.py:151 */
#define ARD_ACT_RELU 2  /* model.py:541 */
#define ARD_ACT_GELU_F16 3 /* same GELU evaluated in packed fp16; the 16-bit output then holds fp16 (feeds ard_gemm_f16) */

#define ARD_MAX_LAYERS 4
#define ARD_CLIP_SAMPLES 480000
#define ARD_FRAMES 1001
#define ARD_MEL_BINS 64
#define ARD_WINDOW_TOKENS 64
#define ARD_CLASS_NUM 527

const char* ard_last_error(void);
int ard_version(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Encoder handle: packed weights + workspace for HTSAT_Swin_Transformer (CLAP/src/laion_clap/clap_module/htsat.py:596-994)
 * and CLAP.audio_projection (clap_module/model.py:539-543).
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct ard_handle ard_handle;

typedef struct ard_config {
    int embed_dim;                 /* 96 tiny / 128 base (htsat.py:1004,1017) */
    int depths[ARD_MAX_LAYERS];    /* {2,2,6,2} / {2,2,12,2} */
    int num_heads[ARD_MAX_LAYERS]; /* {4,8,16,32} */
    int joint_dim;                 /* 512 (model.py joint_embed_shape) */
    int enable_fusion;             /* 1: input is mel_fusion (htsat.py:883-894), 0: waveform (htsat.py:896-910) */
} ard_config;

int ard_create(const ard_config* cfg, ard_handle** out);
int ard_destroy(ard_handle* h);

/* Load one tensor of the reference checkpoint by its state_dict key, audio_branch keys un-prefixed
 * ("layers.2.blocks.5.attn.qkv.weight", "bn0.running_var", "logmel_extractor.melW", ...) plus
 * "audio_projection.{0,2}.{weight,bias}". `data` is float32, HOST memory, `numel` elements. Replaces
 * nn.Module.load_state_dict on the audio branch (factory.py:53-70 key layout). Integer buffers
 * (relative_position_index, num_batches_tracked) and attn_mask are derived, not loaded. */
int ard_set_weight(ard_handle* h, const char* key, const float* data, long long numel);
/* Derive packed device forms (bf16 GEMM operands, q-scale folded into qkv, BN0 folded to scale/shift, banded mel
 * filters, FFT window). Must be called after all weights are set / whenever they change. */
int ard_finalize_weights(ard_handle* h, void* stream);

/* ResiDual injection: replaces patch_block_with_residual(block, residual) (src/residual.py:45-100) for block
 * (layer, block). mean[D], basis[K,D] (rows = components, n_components slices rows: src/residual.py:20-26) are
 * float32 HOST pointers. The patched block reproduces the reference's doubled shortcut/FFN (src/residual.py:91-96). */
int ard_set_block_residual(ard_handle* h, int layer, int block, const float* mean, const float* basis, int K, int D);
int ard_clear_block_residual(ard_handle* h, int layer, int block);
/* lambda = ResiDual.learnable [K] (src/residual.py:27), float32 DEVICE pointer; re-derives the fused
 * projection  W' = M W_proj, b' = (b_proj - mean) M  with  M = B^T diag(lambda) B. */
int ard_set_block_lambda(ard_handle* h, int layer, int block, const float* lambda_dev, void* stream);
/* Same for every patched block of `layer` at once, when they share one ResiDual as setup_residual_htsat builds them
 * (src/residual.py:170-186: one ResiDual per layer, patched into each of its blocks): M is formed once per layer and the
 * blocks' folds run batched. ARD_ERR_STATE if the blocks carry different bases / means (then set them block by block). */
int ard_set_layer_lambda(ard_handle* h, int layer, const float* lambda_dev, void* stream);

typedef struct ard_forward_args {
    const float* waveform;   /* device [B, 480000] fp32 (non-fusion route) */
    const float* mel_fusion; /* device [B, 4, 1001, 64] fp32 (fusion route; only channel 0 is consumed, htsat.py:110-113) */
    int B;
    int quantize;            /* 1: apply quantize_tensor (src/residual.py:210-212) to the waveform on device first */
    float* embedding;        /* device [B, 8*embed_dim]        output_dict['embedding'] (htsat.py:810-811,829) */
    float* audio_embed;      /* device [B, joint_dim] or NULL  CLAP.get_audio_embedding (model.py:739-741) */
    float* layers_residuals[ARD_MAX_LAYERS]; /* device [B, depth_l*T_l, C_l] or NULL  (htsat.py:596,831) */
    float* layers_attention[ARD_MAX_LAYERS]; /* device [B*nW_l, nH_l, 64, 64] or NULL  block-mean (htsat.py:589-595,830) */
    float* framewise_output; /* device [B, 1024, 527] or NULL (htsat.py:818,826) */
    float* clipwise_output;  /* device [B, 527] or NULL (htsat.py:820-821,827) */
    float* fine_grained_embedding; /* device [B, 1024, 8*embed_dim] or NULL (htsat.py:807-808,828) */
    int save_for_backward;   /* 1: keep the activations ard_encoder_backward needs (training step, src/training.py:24-32) */
    float* head_outputs[ARD_MAX_LAYERS];     /* device [depth_l, B*nW_l, nH_l, 64, hd] or NULL: the per-head `attn @ v` temporary of
                                              * WindowAttention.forward (htsat.py:354) of every block, window order of that block
                                              * (shifted blocks: windows of the rolled image), before transpose / proj */
    int precision;           /* 0: bf16/fp16 tensor-core operands (rel. err <= 1e-2); 1: fp32-grade (3-term split-bf16 GEMMs, fp32
                              * attention; rel. err <= 1e-4 vs the reference's fp32 arithmetic, hook.py:40). With save_for_backward,
                              * the precision of the training step: ard_encoder_backward runs at the precision of the saved forward. */
} ard_forward_args;

/* HTSAT_Swin_Transformer.forward (htsat.py:881-994) in eval mode + optional audio_projection/normalize. */
int ard_encoder_forward(ard_handle* h, const ard_forward_args* args, void* stream);

/* Backward of the last ard_encoder_forward(save_for_backward=1) on this handle: what loss.backward() (src/training.py:30-32)
 * computes for the only trainable tensors of setup_residual_htsat (src/residual.py:199-201): the ResiDual `learnable`
 * vectors. The encoder is frozen and in eval mode (src/training.py:105-108), so no weight gradients exist.
 * It runs at the precision of that forward: bf16 tensor-core dgrads (precision 0), or fp32-grade (precision 1: 3-term
 * split-bf16 dgrads, fp32 attention backward / gelu' / LayerNorm backward; rel. err <= 1e-4 vs the reference's fp32 autograd).
 * Inputs are dL/d(audio_embed) and/or dL/d(embedding) (the other output keys: ard_encoder_backward_outputs); grad_lambda[l] (device [K_l] fp32, required for every layer that
 * carries a ResiDual) is OVERWRITTEN with the gradient summed over the layer's patched blocks, which share one
 * ResiDual module in the reference (src/residual.py:186-197). */
typedef struct ard_backward_args {
    int B;
    const float* grad_audio_embed;           /* device [B, joint_dim] or NULL */
    const float* grad_embedding;             /* device [B, 8*embed_dim] or NULL */
    float* grad_lambda[ARD_MAX_LAYERS];      /* device [K_l] fp32 or NULL */
    long long generation;                    /* ard_tape_generation() read right after the forward this backward belongs to; a
                                              * different saved forward on the handle since then -> ARD_ERR_STATE. 0: unchecked */
} ard_backward_args;
int ard_encoder_backward(ard_handle* h, const ard_backward_args* args, void* stream);
/* Gradients of the other keys of output_dict (htsat.py:825-832) for ard_encoder_backward_outputs; every one of them is
 * differentiable w.r.t. ResiDual.learnable in the reference (htsat.py:797-832, src/residual.py:58-98). All device fp32, NULL when
 * the loss does not use that output. The tail keys need a saved forward that computed them (ARD_ERR_STATE otherwise). */
typedef struct ard_output_grads {
    const float* grad_framewise_output;       /* [B, 1024, 527]          sigmoid(tscam_conv) repeated x32, htsat.py:813-818 */
    const float* grad_clipwise_output;        /* [B, 527]                sigmoid(mean_t tscam_conv), htsat.py:820-821 */
    const float* grad_fine_grained_embedding; /* [B, 1024, 8*embed_dim]  frequency-bin mean repeated x32, htsat.py:807-808 */
    const float* grad_layers_residuals[ARD_MAX_LAYERS]; /* [B, depth_l*T_l, C_l]: block b's residual_x (post-ResiDual r of a patched
                                               * block, src/residual.py:88-89; the projected attention branch of a plain one,
                                               * htsat.py:476) at rows b*T_l .. (b+1)*T_l of each clip (htsat.py:589-596) */
    const float* grad_layers_attention[ARD_MAX_LAYERS]; /* [B*nW_l, nH_l, 64, 64] block-mean maps (htsat.py:589-595): every
                                               * block's probabilities receive grad / depth_l, in that block's window order */
} ard_output_grads;
/* ard_encoder_backward with the gradients of the other output_dict keys added to the loss (outs may be NULL: then it is exactly
 * ard_encoder_backward). At least one gradient in args or outs is required. The walk starts at the highest block a given gradient
 * reaches (a loss on layers_residuals[1] alone never touches stages 2-3 or the tail); grad_lambda of a layer no given gradient
 * reaches is written with zeros. */
int ard_encoder_backward_outputs(ard_handle* h, const ard_backward_args* args, const ard_output_grads* outs, void* stream);
/* Op-level tail backward (the tail part of ard_encoder_backward_outputs, on the handle's tscam_conv weights): grad_normed
 * [B, 64, 8*embed_dim] = dL / d(final LayerNorm output) for the loss terms given (each NULL when unused): framewise / clipwise
 * through y = tscam_conv pre-activation [B*32, ldy] fp32 (ldy >= 527, column o of row b*32+t = y[b, o, t]), fine-grained, and
 * grad_embedding [B, 8*embed_dim] (the token mean). precision 0: bf16 tensor-core dgrad; 1: 3-term split-bf16 dgrad. */
int ard_tail_backward(ard_handle* h, const float* y, int ldy, const float* grad_framewise, const float* grad_clipwise, const float* grad_fine,
                      const float* grad_embedding, int B, int precision, float* grad_normed, void* stream);
/* Serial number of the last ard_encoder_forward(save_for_backward=1) on this handle (0: none). The handle keeps ONE tape:
 * a second training forward overwrites it, and a backward carrying the older number is refused instead of silently using
 * the newer activations. */
long long ard_tape_generation(const ard_handle* h);

/* SwinTransformerBlock.forward (htsat.py:439-482) or the ResiDual-patched forward (src/residual.py:58-98) of block
 * (layer, block) on x[B, T_l, C_l] fp32 device. Outputs (device, fp32): x_out [B,T,C]; attn [B*nW,nH,64,64] or NULL;
 * residual_x [B,T,C] or NULL. x_out may alias x_in. */
int ard_block_forward(ard_handle* h, int layer, int block, const float* x_in, int B, float* x_out, float* attn, float* residual_x,
                      void* stream);

/* The attention half of a Swin block as ONE kernel (the window-resident tcgen05 attention block, 96-channel stage):
 * x_out = x + proj'(WindowAttention(norm1(x))) with roll / window_partition / window_reverse as address arithmetic
 * (htsat.py:449-476; proj' carries the ResiDual fold of src/residual.py:88-92 when the block is patched). x_in, x_out
 * [B, T_l, C_l] fp32 device. ARD_ERR_NOTIMPL for layers the kernel does not cover (the encoder uses the unfused chain there). */
int ard_attention_block(ard_handle* h, int layer, int block, const float* x_in, int B, float* x_out, void* stream);

/* Bytes of device workspace the handle currently holds (grown on demand by forward calls). */
long long ard_workspace_bytes(const ard_handle* h);
/* Number of kernels launched by the last ard_encoder_forward / ard_block_forward on this handle. */
int ard_last_launch_count(const ard_handle* h);
/* Process-wide count of kernels this library launched since the last reset (forward, backward, folds, statistics). */
int ard_launch_counter_reset(void);
long long ard_launch_counter_read(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Op-level entry points (the kernels behind the handle; also what the parity tests drive directly)
 * ------------------------------------------------------------------------------------------------------------------ */
/* out[M,N] = act(A[M,K] W[N,K]^T + bias) (+ resid1 + resid2); A, W bf16 device; out bf16 or fp32.  nn.Linear semantics. */
int ard_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_is_bf16, int M, int N,
                  int K, const float* bias, int act, const float* resid1, long long ldr1, const float* resid2, long long ldr2,
                  void* stream);
/* Two contractions of one shape meeting in the epilogue (training backward; bf16 operands, bf16 [M,N] output):
 *   acc1 = A1[M,K] W1[N,K]^T, acc2 = A2[M,K] W2[N,K]^T
 *   mode 0: out = acc1 * gelu'(acc2 + vec1)   - FFN backward dh = (g W2) * gelu'(fc1(norm2(x))), autograd of Mlp htsat.py:146-164
 *   mode 1: dlam[n] += sum_m (acc1 + vec1) * acc2 for n < Kvalid, out = acc2 * vec2[n]
 *           - ResiDual backward, autograd of src/residual.py:37-40: coef = x_proj, acc2 = dL/d x_scaled, vec2 = learnable */
int ard_gemm_dual(int mode, const void* A1, long long lda1, const void* W1, long long ldw1, const void* A2, long long lda2, const void* W2,
                  long long ldw2, void* out, long long ldo, int M, int N, int K, const float* vec1, const float* vec2, float* dlam, int Kvalid,
                  void* stream);
/* Same contraction with fp16 A and W operands (fp32 accumulation): the fc2 GEMM, whose input is the fp16 GELU output. */
int ard_gemm_f16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_is_bf16, int M, int N,
                 int K, const float* bias, int act, const float* resid1, long long ldr1, const float* resid2, long long ldr2,
                 void* stream);
/* Whole FFN of a 96-channel Swin block in one kernel (htsat.py:479-480; src/residual.py:93-96):
 * out[M,96] = x + fc2(gelu(fc1(LayerNorm(x; gamma, beta)))) (+ resid2). x, out, resid2 fp32 device (out may alias x);
 * w1 [384,96] bf16, w2 [96,384] fp16 (the hidden activation is fp16), device; b1 [384], b2 [96] fp32 device. */
int ard_ffn_fused_96(const float* x, const float* resid2, float* out, long long M, const float* gamma, const float* beta, const void* w1_bf16,
                     const float* b1, const void* w2_f16, const float* b2, void* stream);
/* The same FFN for the 192- and 384-channel stages (C = 192 | 384): w1 [4C,C] bf16, w2 [C,4C] fp16, streamed from L2 per
 * 128-token tile. b1_half = 0.5 * fc1 bias [4C] (the packed-fp16 GELU is evaluated on x / 2). */
int ard_ffn_fused_wide(const float* x, const float* resid2, float* out, long long M, int C, const float* gamma, const float* beta,
                       const void* w1_bf16, const float* b1_half, const void* w2_f16, const float* b2, void* stream);
/* norm1 + qkv projection of a 96-channel Swin block in one kernel (htsat.py:449 + :329): qkv[M,288] bf16 =
 * LayerNorm(x[M,96]; gamma, beta) w^T + bias, w [288,96] bf16 (q rows pre-scaled by head_dim^-0.5), all device pointers. */
int ard_ln_qkv_96(const float* x, const float* gamma, const float* beta, const void* w_bf16, const float* bias, void* qkv_bf16, long long M,
                  void* stream);
/* nn.LayerNorm(C, eps=1e-5) over x[rows, C] fp32 -> bf16 (htsat.py:449,479 norm1/norm2). */
int ard_layernorm_bf16(const float* x, const float* gamma, const float* beta, void* out_bf16, long long rows, int C, void* stream);
/* Shifted-window attention core of WindowAttention.forward (htsat.py:326-352) incl. roll/partition/reverse addressing
 * (htsat.py:452-474): qkv bf16 [B*H*W, 3C] in token order (q pre-scaled) -> out bf16 [B*H*W, C] in token order.
 * attn (optional fp32 [B*nW, nH, 64, 64]) receives attn_scale * softmax probabilities (+= if accumulate). */
int ard_window_attention(const void* qkv_bf16, void* out_bf16, const float* bias_table, float* attn, float attn_scale, int accumulate,
                         int B, int H, int W, int C, int nH, int shift, void* stream);
/* fp32 -> bf16 conversion with scale (device). */
/* Backward of ard_window_attention w.r.t. qkv (autograd of htsat.py:326-352): dqkv [B*H*W, 3C] bf16 token order from
 * dout [B*H*W, C] bf16; the probabilities are recomputed from qkv. */
int ard_window_attention_bwd(const void* qkv_bf16, const void* dout_bf16, void* dqkv_bf16, const float* bias_table, int B, int H, int W, int C,
                             int nH, int shift, void* stream);
/* The same backward in fp32 (fp32 CUDA cores; backward of the fp32-grade mode's attention core): qkv [B*H*W, 3C] fp32 token
 * order (q pre-scaled), dout [B*H*W, C] fp32 -> dqkv [B*H*W, 3C] fp32. H == W, head dim C/nH of 24 or 32; no shift when H == 8. */
int ard_window_attention_f32_bwd(const float* qkv_f32, const float* dout_f32, float* dqkv_f32, const float* bias_table, int B, int H, int W,
                                 int C, int nH, int shift, void* stream);
/* The two backwards above with a gradient w.r.t. the attention probabilities as well (a loss on the captured maps,
 * layers_attention = the block mean of BasicLayer.forward, htsat.py:589-595): dP = dO V^T + pscale * pgrad before the softmax
 * backward. pgrad fp32 [B*nW, nH, 64, 64], window order of the block (shifted blocks: windows of the rolled image). */
int ard_window_attention_bwd_pgrad(const void* qkv_bf16, const void* dout_bf16, const float* pgrad, float pscale, void* dqkv_bf16,
                                   const float* bias_table, int B, int H, int W, int C, int nH, int shift, void* stream);
int ard_window_attention_f32_bwd_pgrad(const float* qkv_f32, const float* dout_f32, const float* pgrad, float pscale, float* dqkv_f32,
                                       const float* bias_table, int B, int H, int W, int C, int nH, int shift, void* stream);
/* Backward of nn.LayerNorm over the last dim: grad_in = (add ? add : 0) + dLN(x)^T grad_out; all fp32 [rows, C]. */
int ard_layernorm_bwd(const float* x, const float* grad_out, const float* gamma, const float* add, float* grad_in, long long rows, int C,
                      void* stream);

int ard_f32_to_bf16(const float* in, void* out_bf16, long long n, float scale, void* stream);
/* quantize_tensor (src/residual.py:210-212): clamp, *32767, truncate to int16, /32767; in place allowed. */
int ard_quantize_waveform(const float* in, float* out, long long n, void* stream);

/* Spectrogram + LogmelFilterBank + bn0 (htsat.py:898-902) on device: wave [B, n_samples] -> out [B, 1001, 64]
 * (bn0 applied iff apply_bn). Uses the handle's window / mel filters / BN statistics. */
int ard_logmel(ard_handle* h, const float* wave, int B, int n_samples, int apply_bn, int quantize, float* out, void* stream);

/* bn0 + reshape_wav2img + PatchEmbed (proj conv 4x4/4 + LayerNorm) (htsat.py:900-902, :848-863, :136-143) on a log-mel
 * [B, 1001, 64] (before bn0): out [B, 4096, embed_dim] fp32 = the residual stream entering layer 0. */
int ard_patch_embed(ard_handle* h, const float* logmel, int B, float* out, void* stream);

/* Fusion featuriser: get_mel (training/data.py:363-399: torchaudio MelSpectrogram n_fft 1024 / hop 480 / htk / norm=None +
 * AmplitudeToDB(top_db=None)) for a batch, stacked 4x as get_audio_features does for clips <= 10 s (data.py:497-501):
 * wave [B, n_samples] -> out [B, 4, n_samples/480+1, 64]. Needs "fusion_featuriser.melW" [513,64] and
 * "fusion_featuriser.window" [1024] to have been set with ard_set_weight. */
int ard_fusion_mel(ard_handle* h, const float* wave, int B, int n_samples, int quantize, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Standalone ResiDual module (ResiDual.forward, src/residual.py:29-42) and its autograd: all pointers device fp32.
 *   forward : out[rows,D] = ((x - mean) basis^T * lam) basis           basis [K,D], lam [K], mean [D]
 *   backward: dx[rows,D] = ((g basis^T) * lam) basis (or NULL); dlam[K] += sum_rows ((x - mean) basis^T) * (g basis^T) (or NULL).
 * The contractions run on the tcgen05 GEMM with bf16 operands (fp32 accumulation). Uses per-process scratch: one caller at a time.
 * ------------------------------------------------------------------------------------------------------------------ */
int ard_residual_forward(const float* x, const float* mean, const float* basis, const float* lam, float* out, long long rows, int D, int K,
                         void* stream);
int ard_residual_backward(const float* x, const float* g, const float* mean, const float* basis, const float* lam, float* dx, float* dlam,
                          long long rows, int D, int K, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Classification head on the joint embedding: zero-shot similarities  emb @ text_embeds^T  (src/training.py:28,
 * src/evaluation.py:98) and the linear probe nn.Linear(512, n_classes) (src/linear.py:23-32), CrossEntropyLoss (mean) and
 * their backward (src/training.py:29-31, src/linear.py:43-45). All device fp32; labels int64 device.
 *   ard_head_forward : logits[B,N] = emb[B,J] W[N,J]^T (+ bias[N])
 *   ard_ce_forward   : loss[0] = mean_b( logsumexp(logits_b) - logits_b[label_b] ); dlogits[B,N] = (softmax - onehot) / B (or NULL)
 *   ard_head_backward: d_emb[B,J] = dlogits W;  dW[N,J] = dlogits^T emb;  db[N] = colsum(dlogits)   (each may be NULL)
 * ------------------------------------------------------------------------------------------------------------------ */
int ard_head_forward(const float* emb, const float* W, const float* bias, int B, int N, int J, float* logits, void* stream);
int ard_ce_forward(const float* logits, const long long* labels, int B, int N, float* loss, float* dlogits, void* stream);
int ard_head_backward(const float* dlogits, const float* emb, const float* W, int B, int N, int J, float* d_emb, float* dW, float* db,
                      void* stream);
/* Evaluation reductions on device (the numbers visualize_eval_metrics prints, src/evaluation.py:159-177): for scores[n,C] and
 * int64 targets[n]: counts[0] += #(argmax == target), counts[1] += #(target within the k largest scores, ties ordered as
 * sklearn.top_k_accuracy_score does: of equal scores the higher class index ranks first), cm[C,C] (int64, rows = true class) += 1 at
 * (target, argmax), preds[n] (int64, or NULL) = argmax (first maximal index, as torch.argmax). counts int64 [2] device. */
int ard_eval_metrics(const float* scores, const long long* targets, long long n, int C, int k, long long* counts, long long* cm,
                     long long* preds, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Batched featuriser (replaces the per-clip loop hook.py:175-188 + get_audio_features data.py:466-496 for clips <= max_len):
 * `flat` holds B clips back to back (device, fp32 or int16 PCM), clip b = flat[offsets[b] .. offsets[b]+lengths[b]);
 * (offsets = lengths = NULL: dense [B, max_len] input). out[B, max_len] fp32. mode 0 repeatpad (repeat int(max_len/n) times, zero-pad the rest), 1 pad (zeros), 2 repeat (tile and
 * cut). src_is_pcm16: samples are int16 and are first mapped through int16_to_float32 (data.py:93-94: x / 32767.0).
 * quantize: apply the int16 round trip (data.py:97-99 then :93-94; hook.py:177-179) to float samples on the way.
 * ------------------------------------------------------------------------------------------------------------------ */
int ard_fill_clips(const void* flat, int src_is_pcm16, const long long* offsets, const int* lengths, int B, int max_len, int mode,
                   int quantize, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * PCA sufficient statistics (replaces IncrementalPCA.partial_fit in compute_pca_components, src/residual.py:137-138):
 * accumulates sum[D] += sum_r x[r], sumsq[D,D] += x^T x in float64 on device (the caller counts n). x fp32 [rows, D]
 * device, D a multiple of 4. X^T X runs on the tcgen05 GEMM with x split into two bf16 terms (fp32-grade products,
 * fp32 accumulation per chunk of samples, fp64 across chunks). Uses per-process device scratch: one caller at a time.
 * The _strided form reads rows `ldx` floats apart (e.g. one head's maps out of layers_attention [B*nW, nH, 64, 64],
 * src/analyze_attention.py:41-49, without a gather copy).
 * ------------------------------------------------------------------------------------------------------------------ */
int ard_stats_accumulate(const float* x, long long rows, int D, double* sum, double* sumsq, void* stream);
int ard_stats_accumulate_strided(const float* x, long long rows, long long ldx, int D, double* sum, double* sumsq, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Eigenvalues of `batch` symmetric matrices A[b] (fp64 device, D x D row-major, matrix b at A + b*stride; the lower triangle
 * is read, A is overwritten). w [batch, D] fp64 device, ascending per matrix. work: device scratch of at least
 * ard_sym_eigvals_workspace(D, batch) bytes. Replaces the eigen-solve behind run_PCA's per-head spectra, src/analyze_attention.py:13-59.
 * Blocked Householder tridiagonalisation (dsytrd) + Sturm bisection (dstebz), every launch covering the whole batch; asynchronous
 * on `stream`. ARD_ERR_SHAPE (before any device work): D < 1, batch < 1 or > 65535, stride < D*D, a NULL pointer, a workspace
 * that is too small.
 * ------------------------------------------------------------------------------------------------------------------ */
long long ard_sym_eigvals_workspace(int D, int batch);
int ard_sym_eigvals(double* A, long long stride, int D, int batch, double* w, void* work, long long work_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Eigenvalues and eigenvectors of `batch` symmetric matrices A[b], laid out as for ard_sym_eigvals (lower triangle read, A
 * overwritten). w [batch, D] fp64 device, ascending, bitwise identical to ard_sym_eigvals on the same input (same reduction and
 * bisection). Z[b] at Z + b*zstride: row-major D x D, row m the unit eigenvector of w[b][m]. info [batch] device int: 0, or the
 * number of off-diagonals the tridiagonal QL iteration left unconverged after 30 D sweeps (then Z[b] is not to be used). work:
 * device scratch of at least ard_sym_eigh_workspace(D, batch) bytes (it holds a D x D matrix per batch entry). The eigen-solve
 * behind compute_pca_components (src/residual.py:103-159) and run_PCA's per-head components (src/analyze_attention.py:13-59).
 * Householder tridiagonalisation keeping its reflectors (dsytrd), Sturm bisection (dstebz), implicit QL with the rotations
 * accumulated on the device (tql2), blocked back-transformation (dlarft / dlarfb); asynchronous on `stream`. ARD_ERR_SHAPE
 * (before any device work): every case of ard_sym_eigvals, a NULL Z or info, zstride < D*D, D > 12288.
 * ------------------------------------------------------------------------------------------------------------------ */
long long ard_sym_eigh_workspace(int D, int batch);
int ard_sym_eigh(double* A, long long stride, int D, int batch, double* w, double* Z, long long zstride, int* info,
                 void* work, long long work_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Measurement support (bench.py): per-kernel-class device time. Classes: 0 tcgen05 GEMM, 1 window attention,
 * 2 LayerNorm/merge, 3 front end (STFT/log-mel/patch-embed), 4 heads, 5 other, 6 fused FFN. While enabled every launch is bracketed
 * by CUDA events on its stream; ard_profile_read synchronises, sums elapsed ms / algorithmic flops / algorithmic bytes /
 * launch counts per class since the last read, and clears the records.
 * ------------------------------------------------------------------------------------------------------------------ */
int ard_profile_enable(int on);
int ard_profile_read(double* ms, double* flops, double* bytes, int* launches, int nclass);

#ifdef __cplusplus
}
#endif
#endif /* ARD_H_ */
