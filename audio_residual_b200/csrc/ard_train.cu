// Training path of libard_b200.so: the layout of what the forward keeps for the backward, and the backward schedule that
// produces the gradient of a loss on audio_embed / embedding / the tail keys (framewise, clipwise, fine-grained) / layers_residuals
// w.r.t. every ResiDual `learnable` vector (lambda). The training
// forward is the inference block schedule itself (run_block in ard_api.cu, run_block_fp32 in fp32_mode.cu) pointed at the
// block's tape slots instead of the workspace, so it computes bit for bit what inference computes.
//
// Reference: train_one_epoch  src/training.py:18-37 (loss.backward() through the frozen, eval-mode encoder into
// ResiDual.learnable, src/residual.py:26-27,39) with the patched block forward src/residual.py:58-98.
// Encoder weights are frozen (src/training.py:105-108), so no weight gradients are formed: every backward GEMM is a dgrad
// (dX = dY W) and runs on the same tcgen05 kernel as the forward with a pre-transposed weight copy.
//
// What a block keeps (the "tape", one arena in HBM sized for the batch):
//   s   fp32 [M,C]   block input (= previous block's output buffer, no copy)
//   x1  fp32 [M,C]   s + r                 (input of the first norm2/FFN)
//   x3  fp32 [M,C]   s + x1 + mlp(n2(x1))  (input of the second norm2/FFN, patched blocks only)
//   qkv bf16 [M,3C], ao bf16 [M,C]  attention input / output in token order (fp32 on the fp32-grade tape, precision = 1)
// LayerNorm outputs, the FFN hidden pre-activation and the attention probabilities are recomputed in the backward.
//
// fp32-grade training (precision = 1): the forward writes the same tape slots with qkv / ao in fp32, and the backward mirrors
// the bf16 schedule step for step with every dgrad a 3-term split-bf16 GEMM (gemm3) and everything between the GEMMs fp32:
// the attention backward on CUDA cores, gelu' and the lambda product writing the split form directly.
#include <string.h>

#include "ard_handle.h"

namespace ard {

// heads.cu
int l2_normalize_bwd(const float* p, const float* g, float* out, int B, int N, cudaStream_t s);
int relu_bwd_mul(float* g, const float* act, long long n, cudaStream_t s);
// rowwise.cu
int merge_layernorm_bwd(const float* x, const float* g, const float* gamma, float* dx, __nv_bfloat16* dx_bf, int B, int H, int W, int C,
                        cudaStream_t s);
int gelu_bwd_mul(__nv_bfloat16* dh, const __nv_bfloat16* hpre, long long n, cudaStream_t s);
int bcast_rows(const float* g, float* out, int B, int T, int C, float scale, cudaStream_t s);
int add_f32(const float* a, const float* b, float* y, __nv_bfloat16* ybf, long long n, cudaStream_t s);

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// Carve the tape: every block's output buffer is the next block's `s`; the last block of a layer writes the PatchMerging input.
// precision 0 keeps qkv / ao in bf16 (20 B per token-channel per block), 1 in fp32 (28 B).
int ensure_tape(ard_handle* h, int B, int precision) {
    if (h->tape_B == B && h->tape_prec == precision && h->tape.p) return 0;
    const size_t act_bytes = precision ? 4 : 2;
    size_t total = 0;
    for (int pass = 0; pass < 2; ++pass) {
        uint8_t* base = h->tape.as<uint8_t>();
        size_t off = 0;
        auto take = [&](size_t bytes) -> void* {
            void* p = pass ? base + off : nullptr;
            off += align256(bytes);
            return p;
        };
        float* cur_in = (float*)take((size_t)B * 4096 * C_of(h, 0) * 4);   // patch-embed output
        for (int l = 0; l < h->nlayers; ++l) {
            const size_t MC = (size_t)B * R_of(l) * R_of(l) * C_of(h, l);
            for (int b = 0; b < h->cfg.depths[l]; ++b) {
                BlockW& bw = h->layers[l].blocks[b];
                bw.t_s = cur_in;
                bw.t_x1 = (float*)take(MC * 4);
                bw.t_x3 = (float*)take(MC * 4);
                void* qkv = take(MC * 3 * act_bytes);
                void* ao = take(MC * act_bytes);
                bw.t_qkv = precision ? nullptr : (__nv_bfloat16*)qkv;
                bw.t_ao = precision ? nullptr : (__nv_bfloat16*)ao;
                bw.t_qkvf = precision ? (float*)qkv : nullptr;
                bw.t_aof = precision ? (float*)ao : nullptr;
                bw.t_out = (float*)take(MC * 4);
                cur_in = bw.t_out;
            }
            if (l < h->nlayers - 1) cur_in = (float*)take(MC / 2 * 4);   // merge output [B, T/4, 2C]
        }
        if (pass == 0) {
            total = off;
            h->tape_B = 0;
            ARD_TRY(h->tape.ensure(total));
        }
    }
    h->tape_B = B;
    h->tape_prec = precision;
    return 0;
}

static int transpose_upload_bf16(DevBuf& dst, const float* w, int rows, int cols, float row_scale_first = 1.0f, int scaled_rows = 0) {
    // w [rows, cols] -> dst [cols, rows] bf16; the first `scaled_rows` rows are multiplied by row_scale_first
    std::vector<__nv_bfloat16> t((size_t)rows * cols);
    for (int r = 0; r < rows; ++r) {
        const float sc = r < scaled_rows ? row_scale_first : 1.0f;
        for (int c = 0; c < cols; ++c) t[(size_t)c * rows + r] = __float2bfloat16_rn(w[(size_t)r * cols + c] * sc);
    }
    return upload(dst, t.data(), t.size() * 2);
}

// The ResiDual and the projection fold for the backward too:  with  Wc = B Wp [K,C],  c0 = B (b_p - mu) [K]
//   coef  = x_proj              = ao Wc^T + c0        (src/residual.py:37-38)
//   d ao  = (gcoef * lambda) Wc                        (src/residual.py:39-40 then the proj Linear)
// Host fp32, rows padded to Kp = K rounded up to 16: wc [Kp, C], c0 [Kp], bpad (the basis) [Kp, C].
static int residual_backward_fold(ard_handle* h, int l, int b, std::vector<float>& wc, std::vector<float>& c0, std::vector<float>& bpad) {
    BlockW& bw = h->layers[l].blocks[b];
    const int C = C_of(h, l), K = bw.K, Kp = (K + 15) & ~15;
    char pfx[64];
    snprintf(pfx, sizeof(pfx), "layers.%d.blocks.%d.", l, b);
    const std::string p(pfx);
    const std::vector<float>* pw = nullptr;
    const std::vector<float>* pb = nullptr;
    ARD_TRY(get(h, p + "attn.proj.weight", (size_t)C * C, &pw));
    ARD_TRY(get(h, p + "attn.proj.bias", C, &pb));
    wc.assign((size_t)Kp * C, 0.f);
    c0.assign(Kp, 0.f);
    bpad.assign((size_t)Kp * C, 0.f);
    for (int k = 0; k < K; ++k) {
        const float* bk = bw.h_basis.data() + (size_t)k * C;
        float* o = wc.data() + (size_t)k * C;
        double acc0 = 0.0;
        for (int c = 0; c < C; ++c) {
            const float bv = bk[c];
            const float* wr = pw->data() + (size_t)c * C;
            for (int j = 0; j < C; ++j) o[j] += bv * wr[j];
            acc0 += (double)bv * ((double)(*pb)[c] - (double)bw.h_mean[c]);
        }
        c0[k] = (float)acc0;
        memcpy(bpad.data() + (size_t)k * C, bk, (size_t)C * 4);
    }
    return 0;
}

static int ensure_backward_weights(ard_handle* h, int l, int b) {
    BlockW& bw = h->layers[l].blocks[b];
    if (bw.bwd_ready) return 0;
    const int C = C_of(h, l), nH = h->cfg.num_heads[l];
    char pfx[64];
    snprintf(pfx, sizeof(pfx), "layers.%d.blocks.%d.", l, b);
    const std::string p(pfx);
    const std::vector<float>* v = nullptr;
    ARD_TRY(get(h, p + "mlp.fc1.weight", (size_t)4 * C * C, &v));
    ARD_TRY(transpose_upload_bf16(bw.fc1_wT, v->data(), 4 * C, C));          // [C, 4C]
    ARD_TRY(get(h, p + "mlp.fc2.weight", (size_t)4 * C * C, &v));
    ARD_TRY(transpose_upload_bf16(bw.fc2_wT, v->data(), C, 4 * C));          // [4C, C]
    ARD_TRY(get(h, p + "attn.qkv.weight", (size_t)3 * C * C, &v));
    ARD_TRY(transpose_upload_bf16(bw.qkv_wT, v->data(), 3 * C, C, 1.0f / sqrtf((float)(C / nH)), C));   // [C, 3C], q rows pre-scaled
    const std::vector<float>* pw = nullptr;
    ARD_TRY(get(h, p + "attn.proj.weight", (size_t)C * C, &pw));
    ARD_TRY(transpose_upload_bf16(bw.proj_wT, pw->data(), C, C));
    if (bw.has_res) {
        const int Kp = (bw.K + 15) & ~15;
        bw.Kp = Kp;
        std::vector<float> wc, c0, bpad;
        ARD_TRY(residual_backward_fold(h, l, b, wc, c0, bpad));
        ARD_TRY(upload_bf16(bw.res_wc, wc));                                   // [Kp, C]
        ARD_TRY(transpose_upload_bf16(bw.res_wcT, wc.data(), Kp, C));          // [C, Kp]
        ARD_TRY(upload_bf16(bw.res_basis_bf16, bpad));                         // [Kp, C]
        ARD_TRY(upload_f32(bw.res_c0, c0));
    }
    bw.bwd_ready = true;
    return 0;
}

// w [rows, cols] (the first `scaled_rows` rows times `scale`) -> split form of w^T: dst [cols, 3 rows] = [W_hi^T | W_lo^T | W_hi^T]
static int transpose_split_upload(DevBuf& dst, DevBuf& scratch, const float* w, int rows, int cols, cudaStream_t s, float scale = 1.0f,
                                  int scaled_rows = 0) {
    std::vector<float> t((size_t)rows * cols);
    for (int r = 0; r < rows; ++r) {
        const float sc = r < scaled_rows ? scale : 1.0f;
        for (int c = 0; c < cols; ++c) t[(size_t)c * rows + r] = w[(size_t)r * cols + c] * sc;
    }
    return split3_weight_host(t, scratch, dst, cols, rows, s);
}

// Split forms of every dgrad weight of the fp32-grade backward, next to the forward's split weights (same invalidation).
static int ensure_backward_weights_fp32(ard_handle* h, Fp32Weights& w, cudaStream_t s) {
    if (w.bwd_epoch == w.epoch) return 0;
    const std::vector<float>* v = nullptr;
    for (int l = 0; l < h->nlayers; ++l) {
        const int C = C_of(h, l), nH = h->cfg.num_heads[l];
        for (int b = 0; b < h->cfg.depths[l]; ++b) {
            BlockW& bw = h->layers[l].blocks[b];
            Fp32BlockW& fw = w.blocks[l][b];
            char pfx[64];
            snprintf(pfx, sizeof(pfx), "layers.%d.blocks.%d.", l, b);
            const std::string p(pfx);
            ARD_TRY(get(h, p + "mlp.fc1.weight", (size_t)4 * C * C, &v));
            ARD_TRY(transpose_split_upload(fw.fc1T3, w.scratch, v->data(), 4 * C, C, s));              // [C, 3*4C]
            ARD_TRY(get(h, p + "mlp.fc2.weight", (size_t)4 * C * C, &v));
            ARD_TRY(transpose_split_upload(fw.fc2T3, w.scratch, v->data(), C, 4 * C, s));              // [4C, 3C]
            ARD_TRY(get(h, p + "attn.qkv.weight", (size_t)3 * C * C, &v));
            ARD_TRY(transpose_split_upload(fw.qkvT3, w.scratch, v->data(), 3 * C, C, s, 1.0f / sqrtf((float)(C / nH)), C));   // [C, 3*3C]
            ARD_TRY(get(h, p + "attn.proj.weight", (size_t)C * C, &v));
            ARD_TRY(transpose_split_upload(fw.projT3, w.scratch, v->data(), C, C, s));                 // [C, 3C]
            if (bw.has_res) {
                const int Kp = (bw.K + 15) & ~15;
                std::vector<float> wc, c0, bpad;
                ARD_TRY(residual_backward_fold(h, l, b, wc, c0, bpad));
                ARD_TRY(split3_weight_host(wc, w.scratch, fw.wc3, Kp, C, s));                          // [Kp, 3C]
                ARD_TRY(transpose_split_upload(fw.wcT3, w.scratch, wc.data(), Kp, C, s));              // [C, 3Kp]
                ARD_TRY(split3_weight_host(bpad, w.scratch, fw.basis3, Kp, C, s));                     // [Kp, 3C]
                ARD_TRY(upload_f32(bw.res_c0, c0));
                bw.Kp = Kp;
            }
        }
        if (l < h->nlayers - 1) {
            char key[64];
            snprintf(key, sizeof(key), "layers.%d.downsample.reduction.weight", l);
            ARD_TRY(get(h, key, (size_t)8 * C * C, &v));
            ARD_TRY(transpose_split_upload(w.mergeT3[l], w.scratch, v->data(), 2 * C, 4 * C, s));      // [4C, 3*2C]
        }
    }
    w.bwd_epoch = w.epoch;
    return 0;
}

// ------------------------------------------------------------------------------------------------ backward schedule
struct BwdBufs {
    float *G, *T, *coef, *gcoef;
    __nv_bfloat16 *XN, *HPRE, *DH, *GB, *GQKV, *GAO, *gsc;
};

// gout = out_scale * gin + d/dx [ mlp(norm2(x)) ]^T gin   (one FFN residual branch; gout may alias gin).
// w.GB must hold bf16(gin) on entry; on exit it holds bf16(gin + branch gradient), the bf16 copy of the un-scaled result.
// ext: a layers_residuals gradient added to that bf16 copy only (the operand of the next dgrad, not the shortcut gradient gout).
static int ffn_backward(ard_handle* h, BlockW& bw, int C, long long M, const float* x, const float* gin, float* gout, float out_scale,
                        const BwdBufs& w, cudaStream_t s, RowAddend ext = RowAddend()) {
    ARD_TRY(layernorm_bf16(x, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), w.XN, M, C, s));
    GemmArgs f;
    if (h->use_dual_gemm && C <= 192) {
        // dh = (g W2) * gelu'(fc1(norm2(x))): both products in one kernel, the re-computed pre-activation never reaches HBM.
        // (C >= 384: a 128 x 128 tile of two K = C products moves 4 x 128 x C operand bytes per 16 K outputs out of L2 -
        //  more than the two separate GEMMs with their wider tiles, which stay.)
        DualArgs d;
        d.A1 = w.GB; d.lda1 = C; d.W1 = bw.fc2_wT.as<__nv_bfloat16>(); d.ldw1 = C;
        d.A2 = w.XN; d.lda2 = C; d.W2 = bw.fc1_w.as<__nv_bfloat16>(); d.ldw2 = C;
        d.vec1 = bw.fc1_b.as<float>(); d.out = w.DH; d.ldo = 4 * C; d.M = (int)M; d.N = 4 * C; d.K = C;
        ARD_TRY(gemm_dual_gelu_bwd(d, h->num_sms, s));
    } else {
    f.A = w.XN; f.lda = C; f.W = bw.fc1_w.as<__nv_bfloat16>(); f.ldw = C; f.out = w.HPRE; f.ldo = 4 * C; f.out_bf16 = 1;
    f.M = (int)M; f.N = 4 * C; f.K = C; f.bias = bw.fc1_b.as<float>();
    ARD_TRY(gemm_bf16(f, h->num_sms, s));                                       // hpre = fc1(norm2(x)), recomputed
    f = GemmArgs();
    f.A = w.GB; f.lda = C; f.W = bw.fc2_wT.as<__nv_bfloat16>(); f.ldw = C; f.out = w.DH; f.ldo = 4 * C; f.out_bf16 = 1;
    f.M = (int)M; f.N = 4 * C; f.K = C; f.mul_gelu_bwd = w.HPRE; f.ld_mul = 4 * C;
    ARD_TRY(gemm_bf16(f, h->num_sms, s));                                       // dh = (g W2) * gelu'(hpre), multiplied in the epilogue
    }
    f = GemmArgs();
    f.A = w.DH; f.lda = 4 * C; f.W = bw.fc1_wT.as<__nv_bfloat16>(); f.ldw = 4 * C; f.out = w.T; f.ldo = C;
    f.M = (int)M; f.N = C; f.K = 4 * C;
    ARD_TRY(gemm_bf16(f, h->num_sms, s));                                       // dn2 = dh W1
    return layernorm_bwd(x, w.T, bw.ln2_g.as<float>(), gin, gout, M, C, s, out_scale, w.GB, ext);   // + LN2'(dn2), and its bf16 copy
}

// G holds dL/d(block output) on entry and dL/d(block input) on exit. `stop_after_lambda`: nothing below this block needs
// a gradient, so the attention / norm1 backward of this block is skipped. `ext`: dL/d residual_x from a loss on layers_residuals
// (src/residual.py:88-92, htsat.py:476-479): it adds to dL/dr only, never to the shortcut gradient dL/ds. `pgrad`: dL/d layers_attention
// (or nullptr), whose mean over the layer's blocks (htsat.py:589-595) gives each block's probabilities pgrad / depth.
static int block_backward(ard_handle* h, int l, int b, int B, float* dlam, bool stop_after_lambda, const BwdBufs& w, cudaStream_t s,
                          RowAddend ext, const float* pgrad) {
    BlockW& bw = h->layers[l].blocks[b];
    const int C = C_of(h, l), R = R_of(l), T = R * R, nH = h->cfg.num_heads[l];
    const long long M = (long long)B * T;
    ARD_TRY(ensure_backward_weights(h, l, b));
    GemmArgs g;
    if (bw.has_res) {
        ARD_TRY(ffn_backward(h, bw, C, M, bw.t_x3, w.G, w.G, 1.0f, w, s));       // G  = dL/dx3, GB = bf16(G)
        // dL/dx1 = dL/dr = G + FFN'(G)   (x3 = s + x2, x2 = x1 + mlp): only its bf16 copy (GB) is needed below, and the
        // shortcut sum dL/ds so far = dL/dx3 + dL/dx1 = 2 G + FFN'(G) is written straight into G
        ARD_TRY(ffn_backward(h, bw, C, M, bw.t_x1, w.G, w.G, 2.0f, w, s, ext));   // GB = bf16(dL/dr + ext)
        const int Kp = bw.Kp;
        const float* lam = bw.lambda_set && bw.lam.p ? bw.lam.as<float>() : bw.lam_ones.as<float>();
        if (h->use_dual_gemm) {
            // coef = x_proj = ao Wc^T + c0 and gcoef = dL/d(x_scaled) = dL/dr B^T meet in the epilogue of one kernel:
            // dlam += colsum(coef * gcoef), gsc = gcoef * lam; neither [M, K] fp32 matrix reaches HBM
            DualArgs d;
            d.A1 = bw.t_ao; d.lda1 = C; d.W1 = bw.res_wc.as<__nv_bfloat16>(); d.ldw1 = C;
            d.A2 = w.GB; d.lda2 = C; d.W2 = bw.res_basis_bf16.as<__nv_bfloat16>(); d.ldw2 = C;
            d.vec1 = bw.res_c0.as<float>(); d.vec2 = lam; d.dlam = dlam; d.Kvalid = bw.K;
            d.out = w.gsc; d.ldo = Kp; d.M = (int)M; d.N = Kp; d.K = C;
            ARD_TRY(gemm_dual_lambda(d, h->num_sms, s));
        } else {
        g.A = bw.t_ao; g.lda = C; g.W = bw.res_wc.as<__nv_bfloat16>(); g.ldw = C; g.out = w.coef; g.ldo = Kp;
        g.M = (int)M; g.N = Kp; g.K = C; g.bias = bw.res_c0.as<float>();
        ARD_TRY(gemm_bf16(g, h->num_sms, s));                                    // coef = x_proj
        g = GemmArgs();
        g.A = w.GB; g.lda = C; g.W = bw.res_basis_bf16.as<__nv_bfloat16>(); g.ldw = C; g.out = w.gcoef; g.ldo = Kp;
        g.M = (int)M; g.N = Kp; g.K = C;
        ARD_TRY(gemm_bf16(g, h->num_sms, s));                                    // gcoef = dL/d(x_scaled) = dL/dr B^T
        ARD_TRY(lambda_grad(w.coef, w.gcoef, lam, dlam, w.gsc, M, bw.K, Kp, s));       // dlam += colsum(coef*gcoef); gsc = gcoef*lam
        }
        if (stop_after_lambda) return 0;
        g = GemmArgs();
        g.A = w.gsc; g.lda = Kp; g.W = bw.res_wcT.as<__nv_bfloat16>(); g.ldw = Kp; g.out = w.GAO; g.ldo = C; g.out_bf16 = 1;
        g.M = (int)M; g.N = C; g.K = Kp;
        ARD_TRY(gemm_bf16(g, h->num_sms, s));                                    // d ao = gsc Wc
    } else {
        ARD_TRY(ffn_backward(h, bw, C, M, bw.t_x1, w.G, w.G, 1.0f, w, s, ext));  // G = dL/dx1 = dL/ds (shortcut), GB = bf16(dL/dr = G + ext)
        if (stop_after_lambda) return 0;
        g.A = w.GB; g.lda = C; g.W = bw.proj_wT.as<__nv_bfloat16>(); g.ldw = C; g.out = w.GAO; g.ldo = C; g.out_bf16 = 1;
        g.M = (int)M; g.N = C; g.K = C;
        ARD_TRY(gemm_bf16(g, h->num_sms, s));                                    // d ao = dL/dr Wp
    }
    AttnArgs a;
    a.qkv = bw.t_qkv; a.bias_table = bw.rpb.as<float>(); a.B = B; a.H = R; a.W = R; a.C = C; a.nH = nH; a.shift = (b % 2 == 0) ? 0 : 4;
    ARD_TRY(window_attention_bwd(a, w.GAO, w.GQKV, s, pgrad, 1.0f / h->cfg.depths[l]));
    g = GemmArgs();
    g.A = w.GQKV; g.lda = 3 * C; g.W = bw.qkv_wT.as<__nv_bfloat16>(); g.ldw = 3 * C; g.out = w.T; g.ldo = C;
    g.M = (int)M; g.N = C; g.K = 3 * C;
    ARD_TRY(gemm_bf16(g, h->num_sms, s));                                        // dn1 = dqkv Wqkv
    return layernorm_bwd(bw.t_s, w.T, bw.ln1_g.as<float>(), w.G, w.G, M, C, s, 1.0f, w.GB);  // G += LN1'(dn1), GB = bf16(G)
}

// ------------------------------------------------------------------------------------------------ fp32-grade backward schedule
// The same steps as ffn_backward / block_backward with every dgrad a split GEMM; no gemm_dual (its epilogues are bf16 /
// packed fp16). A3 (split operands, [M, 12C] bf16), HPRE / GQKV (fp32 [M, 4C]) and GAO (fp32 [M, C]) are the fp32-grade
// forward's workspace, idle once the forward is done.
struct BwdBufs32 {
    float *G, *T, *R, *DH, *HPRE, *GQKV, *GAO, *coef, *gcoef;
    __nv_bfloat16 *A3, *G3;
};

// gout = out_scale * gin + d/dx [ mlp(norm2(x)) ]^T gin   (gout may alias gin)
static int ffn_backward_fp32(ard_handle* h, BlockW& bw, Fp32BlockW& fw, int C, long long M, const float* x, const float* gin, float* gout,
                             float out_scale, const BwdBufs32& w, cudaStream_t s) {
    ARD_TRY(layernorm_split3(x, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), w.A3, M, C, s));
    ARD_TRY(gemm3(w.A3, C, fw.fc13, w.HPRE, 4 * C, M, 4 * C, bw.fc1_b.as<float>(), ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));
    ARD_TRY(split3_act(gin, C, w.G3, M, C, s));                                                       // hpre = fc1(norm2(x)), recomputed
    ARD_TRY(gemm3(w.G3, C, fw.fc2T3, w.DH, 4 * C, M, 4 * C, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));   // g W2
    ARD_TRY(gelu_bwd_split3(w.DH, w.HPRE, w.A3, M, 4 * C, s));                                         // dh = (g W2) * gelu'(hpre)
    ARD_TRY(gemm3(w.A3, 4 * C, fw.fc1T3, w.T, C, M, C, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));       // dn2 = dh W1
    return layernorm_bwd(x, w.T, bw.ln2_g.as<float>(), gin, gout, M, C, s, out_scale, nullptr);       // + LN2'(dn2)
}

static int block_backward_fp32(ard_handle* h, Fp32Weights& fws, int l, int b, int B, float* dlam, bool stop_after_lambda, const BwdBufs32& w,
                               cudaStream_t s, RowAddend ext, const float* pgrad) {
    BlockW& bw = h->layers[l].blocks[b];
    Fp32BlockW& fw = fws.blocks[l][b];
    const int C = C_of(h, l), R = R_of(l), T = R * R, nH = h->cfg.num_heads[l];
    const long long M = (long long)B * T;
    if (bw.has_res) {
        ARD_TRY(ffn_backward_fp32(h, bw, fw, C, M, bw.t_x3, w.G, w.G, 1.0f, w, s));     // G = dL/dx3
        ARD_TRY(ffn_backward_fp32(h, bw, fw, C, M, bw.t_x1, w.G, w.R, 1.0f, w, s));     // R = dL/dx1 = dL/dr = G + FFN'(G)
        ARD_TRY(add_f32(w.G, w.R, w.G, nullptr, M * C, s));                             // dL/ds so far = dL/dx3 + dL/dx1
        const int Kp = bw.Kp;
        const float* lam = bw.lambda_set && bw.lam.p ? bw.lam.as<float>() : bw.lam_ones.as<float>();
        ARD_TRY(split3_act(bw.t_aof, C, w.A3, M, C, s));
        ARD_TRY(gemm3(w.A3, C, fw.wc3, w.coef, Kp, M, Kp, bw.res_c0.as<float>(), ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));   // coef = x_proj
        ARD_TRY(split3_act(w.R, C, w.G3, M, C, s, ext));                                // split(dL/dr + ext)
        ARD_TRY(gemm3(w.G3, C, fw.basis3, w.gcoef, Kp, M, Kp, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));   // gcoef = dL/dr B^T
        ARD_TRY(lambda_grad(w.coef, w.gcoef, lam, dlam, w.A3, M, bw.K, Kp, s, true));   // dlam += colsum(coef*gcoef); A3 = split(gcoef*lam)
        if (stop_after_lambda) return 0;
        ARD_TRY(gemm3(w.A3, Kp, fw.wcT3, w.GAO, C, M, C, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));        // d ao = gsc Wc
    } else {
        ARD_TRY(ffn_backward_fp32(h, bw, fw, C, M, bw.t_x1, w.G, w.G, 1.0f, w, s));     // G = dL/dx1 = dL/ds (shortcut) = dL/dr
        if (stop_after_lambda) return 0;
        ARD_TRY(split3_act(w.G, C, w.G3, M, C, s, ext));                                // split(dL/dr = G + ext)
        ARD_TRY(gemm3(w.G3, C, fw.projT3, w.GAO, C, M, C, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));       // d ao = dL/dr Wp
    }
    ARD_TRY(window_attention_f32_bwd(bw.t_qkvf, w.GAO, w.GQKV, bw.rpb.as<float>(), B, R, C, nH, (b % 2 == 0) ? 0 : 4, s, pgrad,
                                     1.0f / h->cfg.depths[l]));
    ARD_TRY(split3_act(w.GQKV, 3 * C, w.A3, M, 3 * C, s));
    ARD_TRY(gemm3(w.A3, 3 * C, fw.qkvT3, w.T, C, M, C, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));          // dn1 = dqkv Wqkv
    return layernorm_bwd(bw.t_s, w.T, bw.ln1_g.as<float>(), w.G, w.G, M, C, s, 1.0f, nullptr);           // G += LN1'(dn1)
}

// ------------------------------------------------------------------------------------------------ tail backward
// Backward of htsat.py:798-821 (restated at heads.cu tscam_im2col_kernel): the per-token gradient in front of the final LayerNorm,
// out [B, 64, NF] = dL/d normed, from the framewise / clipwise terms (through sigma' of the saved pre-sigmoid y and the tscam conv
// dgrad dA = dY W), the fine-grained term and the token mean of g_emb. Everything but the dgrad is fp32; the dgrad is a bf16
// tcgen05 GEMM, or at fp32 grade (fp32) a split gemm3 against [W_hi^T | W_lo^T | W_hi^T].
int tail_backward(ard_handle* h, const float* y, int ldy, const float* g_frame, const float* g_clip, const float* g_fine, const float* g_emb, int B,
                  bool fp32, float* out, cudaStream_t s) {
    const int NF = C_of(h, h->nlayers - 1);
    float* dA = nullptr;
    if (g_frame || g_clip) {
        if (!h->host.count("tscam_conv.weight")) return set_error(ARD_ERR_STATE, "tscam_conv weights were never set");
        const long long rows = (long long)B * 32;
        ARD_TRY(h->bw_tail_da.ensure((size_t)rows * 6 * NF * 4));
        ARD_TRY(h->bw_tail_dy.ensure((size_t)rows * TSCAM_KP * 2 * (fp32 ? 3 : 1)));
        dA = h->bw_tail_da.as<float>();
        __nv_bfloat16* dY = h->bw_tail_dy.as<__nv_bfloat16>();
        ARD_TRY(tscam_bwd_dy(y, ldy, g_frame, g_clip, dY, TSCAM_KP, B, fp32, s));
        if (fp32) {
            Fp32Weights& fw = h->fp32;
            ARD_TRY(ensure_fp32_weights(h, s));
            if (fw.tscam_epoch != fw.epoch) {   // tscam_conv.weight.view(527, 6C) transposed, K = 527 padded to 528, split: built lazily
                const std::vector<float>* v = nullptr;
                ARD_TRY(get(h, "tscam_conv.weight", (size_t)ARD_CLASS_NUM * NF * 6, &v));
                std::vector<float> wp((size_t)TSCAM_KP * 6 * NF, 0.f);
                memcpy(wp.data(), v->data(), (size_t)ARD_CLASS_NUM * 6 * NF * 4);
                ARD_TRY(transpose_split_upload(fw.tscamT3, fw.scratch, wp.data(), TSCAM_KP, 6 * NF, s));   // [6C, 3*528]
                fw.tscam_epoch = fw.epoch;
            }
            ARD_TRY(gemm3(dY, TSCAM_KP, h->fp32.tscamT3, dA, 6 * NF, rows, 6 * NF, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0,
                          h->num_sms, s));
        } else {
            if (!h->tscam_wT.p) {
                const std::vector<float>* v = nullptr;
                ARD_TRY(get(h, "tscam_conv.weight", (size_t)ARD_CLASS_NUM * NF * 6, &v));
                std::vector<float> wp((size_t)TSCAM_KP * 6 * NF, 0.f);
                memcpy(wp.data(), v->data(), (size_t)ARD_CLASS_NUM * 6 * NF * 4);
                ARD_TRY(transpose_upload_bf16(h->tscam_wT, wp.data(), TSCAM_KP, 6 * NF));   // [6NF, 528]
            }
            GemmArgs g;
            g.A = dY; g.lda = TSCAM_KP; g.W = h->tscam_wT.as<__nv_bfloat16>(); g.ldw = TSCAM_KP; g.out = dA; g.ldo = 6LL * NF;
            g.M = (int)rows; g.N = 6 * NF; g.K = TSCAM_KP;
            ARD_TRY(gemm_bf16(g, h->num_sms, s));                                      // dA = dY W
        }
    }
    return tail_token_grad(g_emb, dA, g_fine, out, B, NF, s);
}

int encoder_backward(ard_handle* h, const ard_backward_args* a, const ard_output_grads* o, cudaStream_t s) {
    const int B = a->B;
    if (h->tape_B <= 0 || h->tape_B != B)
        return set_error(ARD_ERR_STATE, "ard_encoder_backward: no saved forward for batch %d (run ard_encoder_forward with save_for_backward=1)", B);
    if (a->generation != 0 && a->generation != h->tape_gen)
        return set_error(ARD_ERR_STATE, "ard_encoder_backward: the saved activations belong to training forward #%lld, this backward to #%lld "
                                        "(the handle keeps one tape: run forward and backward of a step back to back)", h->tape_gen, a->generation);
    const ard_output_grads none = {};
    if (!o) o = &none;
    const int tail = (o->grad_framewise_output ? TAPE_FRAMEWISE : 0) | (o->grad_clipwise_output ? TAPE_CLIPWISE : 0) |
                     (o->grad_fine_grained_embedding ? TAPE_FINE : 0);
    bool any_cap = false;   // a gradient of a per-layer capture (layers_residuals / layers_attention)
    for (int l = 0; l < h->nlayers; ++l) any_cap = any_cap || o->grad_layers_residuals[l] || o->grad_layers_attention[l];
    const bool head = a->grad_audio_embed || a->grad_embedding || tail;
    if (!head && !any_cap) return set_error(ARD_ERR_SHAPE, "ard_encoder_backward: no output gradient given");
    if (tail & ~h->tape_tail)
        return set_error(ARD_ERR_STATE, "ard_encoder_backward_outputs: a gradient for %s, which the saved forward did not compute (request it "
                                        "in the save_for_backward forward)", (tail & ~h->tape_tail & TAPE_FRAMEWISE) ? "framewise_output" :
                                        (tail & ~h->tape_tail & TAPE_CLIPWISE) ? "clipwise_output" : "fine_grained_embedding");
    const int NF = C_of(h, h->nlayers - 1), J = h->cfg.joint_dim;
    // lowest patched block: nothing below it needs a gradient
    int stop_l = -1, stop_b = -1;
    for (int l = h->nlayers - 1; l >= 0; --l)
        for (int b = h->cfg.depths[l] - 1; b >= 0; --b)
            if (h->layers[l].blocks[b].has_res) { stop_l = l; stop_b = b; }
    for (int l = 0; l < h->nlayers; ++l) {
        int K = 0;
        for (BlockW& bw : h->layers[l].blocks)
            if (bw.has_res) {
                if (K && bw.K != K) return set_error(ARD_ERR_SHAPE, "layer %d: blocks carry ResiDuals of different sizes (%d vs %d)", l, K, bw.K);
                K = bw.K;
            }
        if (K && !a->grad_lambda[l]) return set_error(ARD_ERR_SHAPE, "grad_lambda[%d] is required (layer has ResiDual)", l);
        if (K) ARD_TRY(fill_f32(a->grad_lambda[l], K, 0.f, s));
    }
    // the walk starts at the top of the highest layer a given gradient reaches, with G = 0 above it
    int top_l = h->nlayers - 1;
    if (!head)
        while (!o->grad_layers_residuals[top_l] && !o->grad_layers_attention[top_l]) --top_l;
    if (stop_l < 0 || top_l < stop_l) return 0;
    const bool fp32 = h->tape_prec == 1;
    const size_t MC = (size_t)B * 4096 * h->cfg.embed_dim;
    ARD_TRY(h->bw_g.ensure(MC * 4));
    ARD_TRY(h->bw_t.ensure(MC * 4));
    ARD_TRY(h->bw_small.ensure((size_t)B * (2 * J + NF) * 4 + 1024));
    BwdBufs w;
    BwdBufs32 w32;
    Fp32Weights& fws = h->fp32;
    if (fp32) {
        ARD_TRY(ensure_fp32_weights(h, s));
        ARD_TRY(ensure_backward_weights_fp32(h, fws, s));
        ARD_TRY(fws.qkvf.ensure(MC * 16));
        ARD_TRY(fws.aof.ensure(MC * 4));
        ARD_TRY(fws.s3.ensure(MC * 24));
        ARD_TRY(h->bw_gs.ensure(MC * 4));
        ARD_TRY(h->bw_dh.ensure(MC * 16));
        ARD_TRY(h->bw_g3.ensure(MC * 6));
        ARD_TRY(h->bw_coef.ensure(MC * 4));
        ARD_TRY(h->bw_gcoef.ensure(MC * 4));
        w32.G = h->bw_g.as<float>(); w32.T = h->bw_t.as<float>(); w32.R = h->bw_gs.as<float>(); w32.DH = h->bw_dh.as<float>();
        w32.HPRE = w32.GQKV = fws.qkvf.as<float>(); w32.GAO = fws.aof.as<float>();
        w32.coef = h->bw_coef.as<float>(); w32.gcoef = h->bw_gcoef.as<float>();
        w32.A3 = fws.s3.as<__nv_bfloat16>(); w32.G3 = h->bw_g3.as<__nv_bfloat16>();
    } else {
    ARD_TRY(h->bw_dh.ensure(MC * 4 * 2));
    ARD_TRY(h->bw_gb.ensure(MC * 2));
    if (!h->use_dual_gemm) {   // the fp32 coefficient matrices only exist on the separate-GEMM path
        ARD_TRY(h->bw_coef.ensure(MC * 4));
        ARD_TRY(h->bw_gcoef.ensure(MC * 4));
    }
    ARD_TRY(h->bw_gsc.ensure(MC * 2));
    }
    w.G = h->bw_g.as<float>(); w.T = h->bw_t.as<float>();
    w.coef = h->bw_coef.as<float>(); w.gcoef = h->bw_gcoef.as<float>(); w.gsc = h->bw_gsc.as<__nv_bfloat16>();
    w.XN = h->ws_xn.as<__nv_bfloat16>(); w.HPRE = h->ws_h.as<__nv_bfloat16>(); w.DH = h->bw_dh.as<__nv_bfloat16>();
    w.GB = fp32 ? nullptr : h->bw_gb.as<__nv_bfloat16>(); w.GQKV = h->ws_qkv.as<__nv_bfloat16>(); w.GAO = h->ws_ao.as<__nv_bfloat16>();

    if (head) {
    // ---- head: audio_embed = normalize(W2 relu(W0 emb + b0) + b2)   (model.py:539-543, :739-741)
    float* g_p = h->bw_small.as<float>();
    float* g_h = g_p + (size_t)B * J;
    float* g_emb = g_h + (size_t)B * J;
    if (a->grad_audio_embed) {
        if (!h->p0_w.p) return set_error(ARD_ERR_STATE, "audio_projection weights were never set");
        if (!h->p0_wT.p) {
            const std::vector<float>* v = nullptr;
            ARD_TRY(get(h, "audio_projection.0.weight", (size_t)J * NF, &v));
            std::vector<float> t((size_t)J * NF);
            for (int r = 0; r < J; ++r)
                for (int c = 0; c < NF; ++c) t[(size_t)c * J + r] = (*v)[(size_t)r * NF + c];
            ARD_TRY(upload_f32(h->p0_wT, t));
            ARD_TRY(get(h, "audio_projection.2.weight", (size_t)J * J, &v));
            std::vector<float> t2((size_t)J * J);
            for (int r = 0; r < J; ++r)
                for (int c = 0; c < J; ++c) t2[(size_t)c * J + r] = (*v)[(size_t)r * J + c];
            ARD_TRY(upload_f32(h->p2_wT, t2));
        }
        ARD_TRY(l2_normalize_bwd(h->ws_proj.as<float>(), a->grad_audio_embed, g_p, B, J, s));
        ARD_TRY(linear_small(g_p, J, h->p2_wT.as<float>(), nullptr, g_h, J, B, J, J, ARD_ACT_NONE, s));
        ARD_TRY(relu_bwd_mul(g_h, h->ws_hid.as<float>(), (long long)B * J, s));
        ARD_TRY(linear_small(g_h, J, h->p0_wT.as<float>(), nullptr, g_emb, NF, B, NF, J, ARD_ACT_NONE, s));
        if (a->grad_embedding) ARD_TRY(add_f32(g_emb, a->grad_embedding, g_emb, nullptr, (long long)B * NF, s));
    } else if (!tail) {
        ARD_CUDA(cudaMemcpyAsync(g_emb, a->grad_embedding, (size_t)B * NF * 4, cudaMemcpyDeviceToDevice, s));
    }
    // ---- token mean (+ the tail: tscam head and fine-grained embedding, htsat.py:798-821) + final norm (htsat.py:797, :810-811)
    const LayerW& last = h->layers[h->nlayers - 1];
    if (tail)
        ARD_TRY(tail_backward(h, h->ws_tscam_y.as<float>(), TSCAM_KP, o->grad_framewise_output, o->grad_clipwise_output,
                              o->grad_fine_grained_embedding, a->grad_audio_embed ? g_emb : a->grad_embedding, B, fp32, w.T, s));
    else
        ARD_TRY(bcast_rows(g_emb, w.T, B, 64, NF, 1.0f / 64.0f, s));
    ARD_TRY(layernorm_bwd(last.blocks.back().t_out, w.T, h->norm_g.as<float>(), nullptr, w.G, (long long)B * 64, NF, s, 1.0f, w.GB));
    } else {   // only capture gradients: G = 0 (and its bf16 copy) above the highest of them
        const long long Mt = (long long)B * R_of(top_l) * R_of(top_l) * C_of(h, top_l);
        ARD_TRY(fill_f32(h->bw_g.as<float>(), Mt, 0.f, s));
        if (!fp32) ARD_CUDA(cudaMemsetAsync(w.GB, 0, (size_t)Mt * 2, s));
    }
    // ---- swin stages, top down
    for (int l = top_l; l >= stop_l; --l) {
        const int C = C_of(h, l), R = R_of(l), T = R * R, depth = h->cfg.depths[l];
        for (int b = depth - 1; b >= 0; --b) {
            const bool stop = (l == stop_l && b == stop_b);
            const float* gr = o->grad_layers_residuals[l];
            const RowAddend ext{gr ? gr + (long long)b * T * C : nullptr, T, (long long)depth * T * C};
            const float* pg = o->grad_layers_attention[l];
            if (fp32) ARD_TRY(block_backward_fp32(h, fws, l, b, B, a->grad_lambda[l], stop, w32, s, ext, pg));
            else ARD_TRY(block_backward(h, l, b, B, a->grad_lambda[l], stop, w, s, ext, pg));
            if (stop) return 0;
        }
        if (l > 0) {   // PatchMerging backward: reduction Linear (no bias) dgrad, then gather + LayerNorm(4C) backward
            const int Cp = C / 2, Rp = R * 2;
            const long long Mm = (long long)B * R * R;
            LayerW& lw = h->layers[l - 1];
            if (fp32) {
                ARD_TRY(split3_act(w32.G, C, w32.G3, Mm, C, s));
                ARD_TRY(gemm3(w32.G3, C, fws.mergeT3[l - 1], w32.T, 4 * Cp, Mm, 4 * Cp, nullptr, ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0,
                              h->num_sms, s));
                ARD_TRY(merge_layernorm_bwd(lw.blocks.back().t_out, w32.T, lw.mg_g.as<float>(), w32.G, nullptr, B, Rp, Rp, Cp, s));
                continue;
            }
            if (!lw.mg_wT.p) {
                const std::vector<float>* v = nullptr;
                char key[64];
                snprintf(key, sizeof(key), "layers.%d.downsample.reduction.weight", l - 1);
                ARD_TRY(get(h, key, (size_t)8 * Cp * Cp, &v));
                ARD_TRY(transpose_upload_bf16(lw.mg_wT, v->data(), 2 * Cp, 4 * Cp));   // [4Cp, 2Cp]
            }
            GemmArgs g;   // GB = bf16(G) was written by the last block's norm1 backward
            g.A = w.GB; g.lda = C; g.W = lw.mg_wT.as<__nv_bfloat16>(); g.ldw = C; g.out = w.T; g.ldo = 4 * Cp;
            g.M = (int)Mm; g.N = 4 * Cp; g.K = C;
            ARD_TRY(gemm_bf16(g, h->num_sms, s));
            ARD_TRY(merge_layernorm_bwd(lw.blocks.back().t_out, w.T, lw.mg_g.as<float>(), w.G, w.GB, B, Rp, Rp, Cp, s));
        }
    }
    return 0;
}

}  // namespace ard
