// C ABI of libard_b200.so (see include/ard.h): handle management, weight packing from the reference's state_dict keys,
// the encoder forward schedule, and the op-level entry points.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <string>
#include <vector>

#include "ard_handle.h"

namespace ard {

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static thread_local int g_launches = 0;
static long long g_launch_total = 0;   // process-wide, ard_launch_counter_*

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) {
        if (strstr(what, "launch") != nullptr) { ++g_launches; ++g_launch_total; }
        return 0;
    }
    return set_error(ARD_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
void count_launch(int n) { g_launches += n; g_launch_total += n; }
bool pdl_enabled() {
    // Off by default: measured on B200 (tools/batch_sweep.py) it does not shorten the forward (B = 1: 1.03 vs 1.01 ms, B = 256:
    // 11.99 vs 11.57 ms) - successor CTAs that start early compete with the predecessor's tail for the SMs they share.
    static const bool on = [] { const char* e = getenv("ARD_PDL"); return e != nullptr && atoi(e) != 0; }();
    return on;
}

// ------------------------------------------------------------------------------------------------ profiling
struct ProfRec { int cls; cudaEvent_t a, b; double flops, bytes; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
ProfScope::ProfScope(int cls, cudaStream_t s, double flops, double bytes) : idx(-1), stream(s) {
    if (!g_prof_on) return;
    ProfRec r; r.cls = cls; r.flops = flops; r.bytes = bytes;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, s);
    idx = (int)g_prof.size();
    g_prof.push_back(r);
}
ProfScope::~ProfScope() {
    if (idx >= 0) cudaEventRecord(g_prof[idx].b, stream);
}

}  // namespace ard

using namespace ard;

namespace ard {

int upload(DevBuf& b, const void* src, size_t bytes) {
    ARD_TRY(b.ensure(bytes));
    ARD_CUDA(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
    return 0;
}
int upload_f32(DevBuf& b, const std::vector<float>& v) { return upload(b, v.data(), v.size() * 4); }
int upload_f16(DevBuf& b, const std::vector<float>& v) {
    std::vector<__half> t(v.size());
    for (size_t i = 0; i < v.size(); ++i) t[i] = __float2half_rn(v[i]);
    return upload(b, t.data(), t.size() * 2);
}
int upload_bf16(DevBuf& b, const std::vector<float>& v) {
    std::vector<__nv_bfloat16> t(v.size());
    for (size_t i = 0; i < v.size(); ++i) t[i] = __float2bfloat16_rn(v[i]);
    return upload(b, t.data(), t.size() * 2);
}

int get(const ard_handle* h, const std::string& key, size_t numel, const std::vector<float>** out) {
    auto it = h->host.find(key);
    if (it == h->host.end()) return set_error(ARD_ERR_STATE, "weight '%s' was never set", key.c_str());
    if (it->second.size() != numel)
        return set_error(ARD_ERR_SHAPE, "weight '%s' has %zu elements, expected %zu", key.c_str(), it->second.size(), numel);
    *out = &it->second;
    return 0;
}

static int build_mel_bands(const std::vector<float>& melW, DevBuf& w, DevBuf& st_d, DevBuf& ln_d, int* band_max) {
    std::vector<int> st(64), ln(64);
    int bmax = 1;
    for (int m = 0; m < 64; ++m) {
        int lo = 513, hi = -1;
        for (int k = 0; k < 513; ++k)
            if (melW[k * 64 + m] != 0.0f) { lo = k < lo ? k : lo; hi = k; }
        if (hi < 0) { lo = 0; hi = 0; }
        st[m] = lo; ln[m] = hi - lo + 1;
        bmax = ln[m] > bmax ? ln[m] : bmax;
    }
    std::vector<float> band((size_t)64 * bmax, 0.f);
    for (int m = 0; m < 64; ++m)
        for (int q = 0; q < ln[m]; ++q) band[(size_t)m * bmax + q] = melW[(st[m] + q) * 64 + m];
    *band_max = bmax;
    ARD_TRY(upload_f32(w, band));
    ARD_TRY(upload(st_d, st.data(), 64 * 4));
    ARD_TRY(upload(ln_d, ln.data(), 64 * 4));
    return 0;
}

static int upload_twiddle(ard_handle* h) {
    std::vector<float> tw(2048);
    for (int i = 0; i < 1024; ++i) {
        const double a = -2.0 * M_PI * i / 1024.0;
        tw[2 * i] = (float)cos(a);
        tw[2 * i + 1] = (float)sin(a);
    }
    return upload_f32(h->twiddle, tw);
}

static int finalize(ard_handle* h, cudaStream_t) {
    const ard_config& c = h->cfg;
    const std::vector<float>* v = nullptr;
    const std::vector<float>* v2 = nullptr;
    // ---- front end
    if (!c.enable_fusion) {
        // window = row k=0 of the (cos * window) Conv1d kernel (torchlibrosa STFT: W_real[k, 0, n] = cos(2 pi k n / N) * win[n])
        ARD_TRY(get(h, "spectrogram_extractor.stft.conv_real.weight", 513 * 1024, &v));
        std::vector<float> win(v->begin(), v->begin() + 1024);
        ARD_TRY(upload_f32(h->window, win));
        ARD_TRY(upload_twiddle(h));
        ARD_TRY(get(h, "logmel_extractor.melW", 513 * 64, &v));
        ARD_TRY(build_mel_bands(*v, h->melw, h->mstart, h->mlen, &h->band_max));
    }
    if (h->host.count("fusion_featuriser.melW")) {   // torchaudio MelSpectrogram(htk, norm=None) filters + window of get_mel
        ARD_TRY(upload_twiddle(h));
        ARD_TRY(get(h, "fusion_featuriser.window", 1024, &v));
        ARD_TRY(upload_f32(h->f_window, *v));
        ARD_TRY(get(h, "fusion_featuriser.melW", 513 * 64, &v));
        ARD_TRY(build_mel_bands(*v, h->f_melw, h->f_mstart, h->f_mlen, &h->f_band_max));
    }
    {   // bn0 eval: y = (x - rm) / sqrt(rv + eps) * g + b  ->  scale, shift   (htsat.py:691, :900-902)
        const std::vector<float>*g, *b, *rm, *rv;
        ARD_TRY(get(h, "bn0.weight", 64, &g));
        ARD_TRY(get(h, "bn0.bias", 64, &b));
        ARD_TRY(get(h, "bn0.running_mean", 64, &rm));
        ARD_TRY(get(h, "bn0.running_var", 64, &rv));
        std::vector<float> sc(64), sh(64);
        for (int i = 0; i < 64; ++i) {
            const double s = (double)(*g)[i] / sqrt((double)(*rv)[i] + 1e-5);
            sc[i] = (float)s;
            sh[i] = (float)((double)(*b)[i] - (double)(*rm)[i] * s);
        }
        ARD_TRY(upload_f32(h->bn_scale, sc));
        ARD_TRY(upload_f32(h->bn_shift, sh));
    }
    const int C0 = c.embed_dim;
    ARD_TRY(get(h, "patch_embed.proj.weight", (size_t)C0 * 16, &v)); ARD_TRY(upload_f32(h->pe_w, *v));
    ARD_TRY(get(h, "patch_embed.proj.bias", C0, &v)); ARD_TRY(upload_f32(h->pe_b, *v));
    ARD_TRY(get(h, "patch_embed.norm.weight", C0, &v)); ARD_TRY(upload_f32(h->pe_g, *v));
    ARD_TRY(get(h, "patch_embed.norm.bias", C0, &v)); ARD_TRY(upload_f32(h->pe_beta, *v));
    // ---- swin layers
    for (int l = 0; l < h->nlayers; ++l) {
        const int C = C_of(h, l), nH = c.num_heads[l];
        if (C % nH) return set_error(ARD_ERR_SHAPE, "layer %d: dim %d not divisible by heads %d", l, C, nH);
        const int hd = C / nH;
        const float qscale = 1.0f / sqrtf((float)hd);   // htsat.py:295 head_dim ** -0.5, folded into the q rows
        for (int b = 0; b < c.depths[l]; ++b) {
            BlockW& bw = h->layers[l].blocks[b];
            char pfx[64];
            snprintf(pfx, sizeof(pfx), "layers.%d.blocks.%d.", l, b);
            const std::string p(pfx);
            ARD_TRY(get(h, p + "norm1.weight", C, &v)); ARD_TRY(upload_f32(bw.ln1_g, *v));
            ARD_TRY(get(h, p + "norm1.bias", C, &v)); ARD_TRY(upload_f32(bw.ln1_b, *v));
            ARD_TRY(get(h, p + "norm2.weight", C, &v)); ARD_TRY(upload_f32(bw.ln2_g, *v));
            ARD_TRY(get(h, p + "norm2.bias", C, &v)); ARD_TRY(upload_f32(bw.ln2_b, *v));
            ARD_TRY(get(h, p + "attn.qkv.weight", (size_t)3 * C * C, &v));
            ARD_TRY(get(h, p + "attn.qkv.bias", (size_t)3 * C, &v2));
            {
                std::vector<float> w(*v), bb(*v2);
                for (size_t i = 0; i < (size_t)C * C; ++i) w[i] *= qscale;
                for (int i = 0; i < C; ++i) bb[i] *= qscale;
                ARD_TRY(upload_bf16(bw.qkv_w, w));
                ARD_TRY(upload_f32(bw.qkv_b, bb));
            }
            ARD_TRY(get(h, p + "attn.proj.weight", (size_t)C * C, &v));
            ARD_TRY(upload_bf16(bw.proj_w, *v));
            ARD_TRY(upload_f32(bw.proj_w_f32, *v));
            ARD_TRY(get(h, p + "attn.proj.bias", C, &v)); ARD_TRY(upload_f32(bw.proj_b, *v));
            ARD_TRY(get(h, p + "mlp.fc1.weight", (size_t)4 * C * C, &v)); ARD_TRY(upload_bf16(bw.fc1_w, *v));
            ARD_TRY(get(h, p + "mlp.fc1.bias", (size_t)4 * C, &v)); ARD_TRY(upload_f32(bw.fc1_b, *v));
            {
                std::vector<float> hb(*v);
                for (auto& t : hb) t *= 0.5f;
                ARD_TRY(upload_f32(bw.fc1_b_half, hb));   // ffn_wide's packed GELU takes x / 2
            }
            ARD_TRY(get(h, p + "mlp.fc2.weight", (size_t)4 * C * C, &v)); ARD_TRY(upload_f16(bw.fc2_w, *v));   // hidden activations are fp16
            ARD_TRY(get(h, p + "mlp.fc2.bias", C, &v)); ARD_TRY(upload_f32(bw.fc2_b, *v));
            ARD_TRY(get(h, p + "attn.relative_position_bias_table", (size_t)225 * nH, &v)); ARD_TRY(upload_f32(bw.rpb, *v));
            if (C == 96 && nH == 4) {   // window-resident attention block kernel: per-head padded q/k/v weights + padded projection
                const std::vector<float>*qw, *qb;
                ARD_TRY(get(h, p + "attn.qkv.weight", (size_t)3 * C * C, &qw));
                ARD_TRY(get(h, p + "attn.qkv.bias", (size_t)3 * C, &qb));
                ARD_TRY(attn_block_pack(bw.ab, *qw, *qb, *v, C, nH));
                ARD_TRY(bw.ab.wp_plain.ensure((size_t)C * 128 * 2));
                ARD_TRY(bw.ab.wp_fold.ensure((size_t)C * 128 * 2));
                ARD_TRY(bw.ab.bp_plain.ensure((size_t)C * 4));
                ARD_TRY(bw.ab.bp_fold.ensure((size_t)C * 4));
                ARD_TRY(attn_block_pad_proj(bw.proj_w.as<__nv_bfloat16>(), bw.proj_b.as<float>(), bw.ab.bv.as<float>(), bw.ab.wp_plain.as<__nv_bfloat16>(),
                                            bw.ab.bp_plain.as<float>(), C, nH, nullptr));
            }
            if (bw.has_res) {   // proj bias may have changed: refresh (b_proj - mean) and force a re-fold
                std::vector<float> dm(C);
                const std::vector<float>* pb;
                ARD_TRY(get(h, p + "attn.proj.bias", C, &pb));
                for (int i = 0; i < C; ++i) dm[i] = (*pb)[i] - bw.h_mean[i];
                ARD_TRY(upload_f32(bw.res_dmean, dm));
                bw.lambda_set = false;
            }
            bw.bwd_ready = false;
        }
        if (l < h->nlayers - 1) {
            char pfx[64];
            snprintf(pfx, sizeof(pfx), "layers.%d.downsample.", l);
            const std::string p(pfx);
            ARD_TRY(get(h, p + "norm.weight", (size_t)4 * C, &v)); ARD_TRY(upload_f32(h->layers[l].mg_g, *v));
            ARD_TRY(get(h, p + "norm.bias", (size_t)4 * C, &v)); ARD_TRY(upload_f32(h->layers[l].mg_b, *v));
            ARD_TRY(get(h, p + "reduction.weight", (size_t)8 * C * C, &v)); ARD_TRY(upload_bf16(h->layers[l].mg_w, *v));
        }
    }
    const int NF = C_of(h, h->nlayers - 1);
    ARD_TRY(get(h, "norm.weight", NF, &v)); ARD_TRY(upload_f32(h->norm_g, *v));
    ARD_TRY(get(h, "norm.bias", NF, &v)); ARD_TRY(upload_f32(h->norm_b, *v));
    if (h->host.count("tscam_conv.weight")) {
        ARD_TRY(get(h, "tscam_conv.weight", (size_t)ARD_CLASS_NUM * NF * 6, &v)); ARD_TRY(upload_bf16(h->tscam_w, *v));
        ARD_TRY(get(h, "tscam_conv.bias", ARD_CLASS_NUM, &v)); ARD_TRY(upload_f32(h->tscam_b, *v));
    }
    if (h->host.count("audio_projection.0.weight")) {
        const int J = c.joint_dim;
        ARD_TRY(get(h, "audio_projection.0.weight", (size_t)J * NF, &v)); ARD_TRY(upload_f32(h->p0_w, *v));
        ARD_TRY(get(h, "audio_projection.0.bias", J, &v)); ARD_TRY(upload_f32(h->p0_b, *v));
        ARD_TRY(get(h, "audio_projection.2.weight", (size_t)J * J, &v)); ARD_TRY(upload_f32(h->p2_w, *v));
        ARD_TRY(get(h, "audio_projection.2.bias", J, &v)); ARD_TRY(upload_f32(h->p2_b, *v));
    }
    // transposed copies the backward builds lazily from the host tensors (ard_train.cu) are stale now
    auto drop = [](DevBuf& b) { if (b.p) { cudaFree(b.p); b.p = nullptr; b.bytes = 0; ++alloc_epoch(); } };
    drop(h->p0_wT); drop(h->p2_wT); drop(h->tscam_wT);
    for (LayerW& lw : h->layers) drop(lw.mg_wT);
    h->tape_B = 0;   // activations of a forward run with the old weights must not be back-propagated through the new ones
    h->finalized = true;
    return 0;
}

// ------------------------------------------------------------------------------------------------ forward schedule
int ensure_workspace(ard_handle* h, int B) {
    const size_t MC = (size_t)B * 4096 * h->cfg.embed_dim;   // max over stages of tokens*channels
    ARD_TRY(h->ws_x.ensure(MC * 4));
    ARD_TRY(h->ws_y.ensure(MC * 4));
    ARD_TRY(h->ws_xn.ensure(MC * 2));
    ARD_TRY(h->ws_ao.ensure(MC * 2));
    ARD_TRY(h->ws_qkv.ensure(MC * 3 * 2));
    ARD_TRY(h->ws_h.ensure(MC * 4 * 2));
    return 0;
}

int ensure_fold(ard_handle* h, int l, int b, cudaStream_t s) {
    BlockW& bw = h->layers[l].blocks[b];
    if (!bw.has_res || bw.lambda_set) return 0;
    // learnable initialises to ones (src/residual.py:27)
    const int C = C_of(h, l);
    std::vector<float> ones((bw.K + 15) & ~15, 0.0f);   // padded to the backward GEMMs' K granularity
    for (int i = 0; i < bw.K; ++i) ones[i] = 1.0f;
    ARD_TRY(upload_f32(bw.lam_ones, ones));
    ARD_TRY(residual_fold(bw.proj_w_f32.as<float>(), bw.res_dmean.as<float>(), bw.res_basis.as<float>(), bw.lam_ones.as<float>(), C, bw.K,
                          bw.res_M.as<float>(), bw.proj_w_fold.as<__nv_bfloat16>(), bw.proj_b_fold.as<float>(), s, bw.proj_w_fold_f32.as<float>()));
    if (bw.ab.ready)
        ARD_TRY(attn_block_pad_proj(bw.proj_w_fold.as<__nv_bfloat16>(), bw.proj_b_fold.as<float>(), bw.ab.bv.as<float>(), bw.ab.wp_fold.as<__nv_bfloat16>(),
                                    bw.ab.bp_fold.as<float>(), C, h->cfg.num_heads[l], s));
    bw.lambda_set = true;
    return 0;
}

// Where one block reads and writes. Inference: s = out = X (the residual stream), x1 = x3 = Y (scratch), qkv / ao in the
// workspace. Training (tape): the block's tape slots (ard_train.cu), so the backward finds every intermediate it needs and the
// training forward computes bit for bit what inference does.
struct BlockIO {
    float *s, *x1, *x3, *out;
    __nv_bfloat16 *qkv, *ao;
    bool tape;   // qkv / ao must be materialised (the fused attention block keeps them on chip)
};

// One Swin block: plain htsat.py:439-482, patched src/residual.py:58-98 (doubled shortcut + FFN, SURVEY Q2).
static int run_block(ard_handle* h, int l, int b, int B, const BlockIO& io, float* attn_out, float attn_scale, int attn_acc,
                     float* res_out, long long res_bstride, float* head_tap, cudaStream_t s) {
    BlockW& bw = h->layers[l].blocks[b];
    const int C = C_of(h, l), R = R_of(l), T = R * R, nH = h->cfg.num_heads[l];
    const long long M = (long long)B * T;
    __nv_bfloat16* XN = h->ws_xn.as<__nv_bfloat16>();
    __nv_bfloat16* Hb = h->ws_h.as<__nv_bfloat16>();
    const int shift = (b % 2 == 0) ? 0 : 4;   // htsat.py:563

    GemmArgs g;
    const bool fused_attn = h->use_attn_block && bw.ab.ready && !io.tape && !attn_out && !res_out && !head_tap && (R % 16) == 0;
    if (fused_attn) {
        // norm1 + qkv + window attention + (folded) projection + shortcut in ONE kernel: x1 = s + r. q/k/v, the attention
        // probabilities and the attention output never reach HBM (capture outputs and the tape need them: those calls take the path below)
        ARD_TRY(ensure_fold(h, l, b, s));
        ARD_TRY(attn_block_96(io.s, io.x1, bw.ab, (bw.has_res ? bw.ab.wp_fold : bw.ab.wp_plain).as<__nv_bfloat16>(),
                              (bw.has_res ? bw.ab.bp_fold : bw.ab.bp_plain).as<float>(), bw.ln1_g.as<float>(), bw.ln1_b.as<float>(), B, R, shift,
                              h->num_sms, s));
    } else {
    if (C == 96 && h->use_ln_qkv) {   // norm1 + qkv in one kernel: the bf16 LayerNorm output never reaches HBM
        ARD_TRY(ln_qkv_96(io.s, bw.ln1_g.as<float>(), bw.ln1_b.as<float>(), bw.qkv_w.as<__nv_bfloat16>(), bw.qkv_b.as<float>(), io.qkv, M,
                          h->num_sms, s));
    } else {
        ARD_TRY(layernorm_bf16(io.s, bw.ln1_g.as<float>(), bw.ln1_b.as<float>(), XN, M, C, s));
        g.A = XN; g.lda = C; g.W = bw.qkv_w.as<__nv_bfloat16>(); g.ldw = C; g.out = io.qkv; g.ldo = 3 * C; g.out_bf16 = 1;
        g.M = (int)M; g.N = 3 * C; g.K = C; g.bias = bw.qkv_b.as<float>();
        ARD_TRY(gemm_bf16(g, h->num_sms, s));
    }
    AttnArgs a;
    a.qkv = io.qkv; a.out = io.ao; a.bias_table = bw.rpb.as<float>(); a.attn_mean = attn_out; a.attn_scale = attn_scale; a.attn_accumulate = attn_acc;
    a.B = B; a.H = R; a.W = R; a.C = C; a.nH = nH; a.shift = shift;
    ARD_TRY(window_attention(a, s));
    if (head_tap) ARD_TRY(head_output_tap(io.ao, head_tap, B, R, C, nH, shift, s));   // per-head attn @ v (htsat.py:354)
    // proj (+ folded ResiDual) + shortcut:  x1 = s + r,  aux = r = residual_x
    ARD_TRY(ensure_fold(h, l, b, s));
    g = GemmArgs();
    g.A = io.ao; g.lda = C; g.ldw = C; g.out = io.x1; g.ldo = C; g.M = (int)M; g.N = C; g.K = C;
    if (bw.has_res) { g.W = bw.proj_w_fold.as<__nv_bfloat16>(); g.bias = bw.proj_b_fold.as<float>(); }
    else { g.W = bw.proj_w.as<__nv_bfloat16>(); g.bias = bw.proj_b.as<float>(); }
    g.resid1 = io.s; g.ldr1 = C;
    if (res_out) { g.aux = res_out; g.ld_aux = C; g.aux_T = T; g.aux_bstride = res_bstride; }
    ARD_TRY(gemm_bf16(g, h->num_sms, s));
    }
    // one FFN: out = in + mlp(norm2(in)) (+ r2), the second residual inside the fused kernel or the fc2 epilogue.
    // HTSAT-base widths (C = 128 / 256) are opt-in (ARD_FUSED_FFN_WIDE=3): the kernel passes its parity tests there and is 6 % faster
    // on the base model (24.0 -> 22.6 ms per 256 clips), but with it the FIRST graph executions of a fresh handle faulted
    // ("unspecified launch failure") 6 times in ~260 tries against 0 in ~280 without it; the cause is not found, so the default keeps
    // the base model on the chain that has never faulted. (profiles/r2_summary.md, "Open issue".)
    // ffn_wide (weights streamed from L2) is used where it measures faster than LayerNorm + two GEMMs: both FFNs of the
    // 192-channel stage (217 / 255 us plain / with second residual vs 341 / 339 us at B = 256). At C = 384 (254 vs 200 us: three
    // ring slots cannot cover the L2 latency) the unfused chain stays. ARD_FUSED_FFN_WIDE=2 forces it for C = 384 too (A/B
    // measurements), =0 disables it.
    const bool wide = (C == 192 && h->use_fused_ffn_wide >= 1) || ((C == 128 || C == 256) && h->use_fused_ffn_wide >= 3) ||
                      (C == 384 && h->use_fused_ffn_wide >= 2);
    auto ffn = [&](const float* in, float* out, const float* r2) -> int {
        if (C == 96 && h->use_fused_ffn)   // whole FFN in one kernel, hidden activation never leaves the SM
            return ffn_fused_96(in, r2, out, M, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), bw.fc1_w.as<__nv_bfloat16>(), bw.fc1_b.as<float>(),
                                bw.fc2_w.as<__half>(), bw.fc2_b.as<float>(), h->num_sms, s);
        if (wide)                          // same, weights streamed from L2
            return ffn_fused_wide(in, r2, out, M, C, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), bw.fc1_w.as<__nv_bfloat16>(),
                                  bw.fc1_b_half.as<float>(), bw.fc2_w.as<__half>(), bw.fc2_b.as<float>(), h->num_sms, s);
        ARD_TRY(layernorm_bf16(in, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), XN, M, C, s));
        GemmArgs f;
        f.A = XN; f.lda = C; f.W = bw.fc1_w.as<__nv_bfloat16>(); f.ldw = C; f.out = Hb; f.ldo = 4 * C; f.out_bf16 = 1;
        f.M = (int)M; f.N = 4 * C; f.K = C; f.bias = bw.fc1_b.as<float>(); f.act = ARD_ACT_GELU; f.out_f16 = 1;
        ARD_TRY(gemm_bf16(f, h->num_sms, s));
        f = GemmArgs();
        f.A = Hb; f.lda = 4 * C; f.W = bw.fc2_w.as<__nv_bfloat16>(); f.ldw = 4 * C; f.out = out; f.ldo = C; f.ab_f16 = 1;
        f.M = (int)M; f.N = C; f.K = 4 * C; f.bias = bw.fc2_b.as<float>();
        f.resid1 = in; f.ldr1 = C; f.resid2 = r2; f.ldr2 = C;   // ((acc + b) + in) + r2
        return gemm_bf16(f, h->num_sms, s);
    };
    if (!bw.has_res) return ffn(io.x1, io.out, nullptr);     // htsat.py:480
    ARD_TRY(ffn(io.x1, io.x3, io.s));                        // x3 = shortcut + (x1 + mlp(norm2(x1)))   src/residual.py:93,95
    return ffn(io.x3, io.out, nullptr);                      // x4 = x3 + mlp(norm2(x3))                src/residual.py:96
}

static int encoder_forward(ard_handle* h, const ard_forward_args* a, cudaStream_t s) {
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    const int B = a->B;
    if (B <= 0) return set_error(ARD_ERR_SHAPE, "batch must be positive (got %d)", B);
    if (!a->embedding) return set_error(ARD_ERR_SHAPE, "embedding output is required");
    if (a->precision != 0 && a->precision != 1) return set_error(ARD_ERR_SHAPE, "precision must be 0 (bf16) or 1 (fp32-grade), got %d", a->precision);
    const bool fp32 = a->precision == 1;
    const int C0 = h->cfg.embed_dim;
    ARD_TRY(ensure_workspace(h, B));
    float* X = h->ws_x.as<float>();
    float* Y = h->ws_y.as<float>();
    const bool train = a->save_for_backward != 0;
    h->tape_B = train ? h->tape_B : 0;   // an inference forward overwrites the head activations the backward would read
    if (train) {
        ARD_TRY(ensure_tape(h, B, a->precision));
        ++h->tape_gen;
        // the tail backward reads this forward's tscam pre-activation (ws_tscam_y), which the next inference forward overwrites
        h->tape_tail = (a->framewise_output ? TAPE_FRAMEWISE : 0) | (a->clipwise_output ? TAPE_CLIPWISE : 0) |
                       (a->fine_grained_embedding ? TAPE_FINE : 0);
        X = h->layers[0].blocks[0].t_s;
    }
    // ---- front end
    if (h->cfg.enable_fusion) {
        if (!a->mel_fusion) return set_error(ARD_ERR_SHAPE, "fusion model expects mel_fusion input");
        ARD_TRY(patch_embed_ln(a->mel_fusion, 4LL * ARD_FRAMES * 64, ARD_FRAMES, h->bn_scale.as<float>(), h->bn_shift.as<float>(),
                               h->pe_w.as<float>(), h->pe_b.as<float>(), h->pe_g.as<float>(), h->pe_beta.as<float>(), X, B, C0, s));
    } else {
        if (!a->waveform) return set_error(ARD_ERR_SHAPE, "non-fusion model expects waveform input");
        ARD_TRY(h->ws_logmel.ensure((size_t)B * ARD_FRAMES * 64 * 4));
        MelBands mb{h->melw.as<float>(), h->mstart.as<int>(), h->mlen.as<int>(), h->band_max};
        ARD_TRY(stft_logmel(a->waveform, B, ARD_CLIP_SAMPLES, h->window.as<float>(), h->twiddle.as<float2>(), mb, nullptr, nullptr,
                            h->ws_logmel.as<float>(), 0, 1, a->quantize, s));
        ARD_TRY(patch_embed_ln(h->ws_logmel.as<float>(), (long long)ARD_FRAMES * 64, ARD_FRAMES, h->bn_scale.as<float>(),
                               h->bn_shift.as<float>(), h->pe_w.as<float>(), h->pe_b.as<float>(), h->pe_g.as<float>(), h->pe_beta.as<float>(),
                               X, B, C0, s));
    }
    // ---- swin stages (fp32-grade: the training forward writes the fp32 tape there)
    if (fp32) ARD_TRY(encoder_stages_fp32(h, a, X, Y, &X, s));
    for (int l = 0; l < h->nlayers && !fp32; ++l) {
        const int C = C_of(h, l), R = R_of(l), T = R * R, depth = h->cfg.depths[l];
        for (int b = 0; b < depth; ++b) {
            float* res = a->layers_residuals[l] ? a->layers_residuals[l] + (long long)b * T * C : nullptr;
            // BasicLayer.forward (htsat.py:589-596): mean of the blocks' maps; residuals concatenated along tokens
            float* tap = a->head_outputs[l] ? a->head_outputs[l] + (long long)b * B * T * C : nullptr;
            const BlockW& bw = h->layers[l].blocks[b];
            const BlockIO io = train ? BlockIO{bw.t_s, bw.t_x1, bw.t_x3, bw.t_out, bw.t_qkv, bw.t_ao, true}
                                     : BlockIO{X, Y, Y, X, h->ws_qkv.as<__nv_bfloat16>(), h->ws_ao.as<__nv_bfloat16>(), false};
            ARD_TRY(run_block(h, l, b, B, io, a->layers_attention[l], 1.0f / depth, b > 0, res, (long long)depth * T, tap, s));
            if (train) X = bw.t_out;
        }
        if (l < h->nlayers - 1) {   // PatchMerging (htsat.py:505-526)
            __nv_bfloat16* Hb = h->ws_h.as<__nv_bfloat16>();
            ARD_TRY(merge_layernorm_bf16(X, h->layers[l].mg_g.as<float>(), h->layers[l].mg_b.as<float>(), Hb, B, R, R, C, s));
            GemmArgs g;
            float* mout = train ? h->layers[l + 1].blocks[0].t_s : Y;
            g.A = Hb; g.lda = 4 * C; g.W = h->layers[l].mg_w.as<__nv_bfloat16>(); g.ldw = 4 * C; g.out = mout; g.ldo = 2 * C;
            g.M = B * (T / 4); g.N = 2 * C; g.K = 4 * C;
            ARD_TRY(gemm_bf16(g, h->num_sms, s));
            if (train) X = mout;
            else { float* t = X; X = Y; Y = t; }
        }
    }
    // ---- tail
    const int NF = C_of(h, h->nlayers - 1);
    const bool need_tscam = a->framewise_output || a->clipwise_output || a->fine_grained_embedding;
    float* normed = nullptr;
    if (need_tscam) {
        ARD_TRY(h->ws_normed.ensure((size_t)B * 64 * NF * 4));
        normed = h->ws_normed.as<float>();
    }
    ARD_TRY(final_norm_mean(X, h->norm_g.as<float>(), h->norm_b.as<float>(), a->embedding, normed, B, 64, NF, s));
    if (a->audio_embed) {
        if (!h->p0_w.p) return set_error(ARD_ERR_STATE, "audio_projection weights were never set");
        const int J = h->cfg.joint_dim;
        ARD_TRY(h->ws_hid.ensure((size_t)B * J * 4));
        ARD_TRY(h->ws_proj.ensure((size_t)B * J * 4));
        ARD_TRY(linear_small(a->embedding, NF, h->p0_w.as<float>(), h->p0_b.as<float>(), h->ws_hid.as<float>(), J, B, J, NF, ARD_ACT_RELU, s));
        ARD_TRY(linear_small(h->ws_hid.as<float>(), J, h->p2_w.as<float>(), h->p2_b.as<float>(), h->ws_proj.as<float>(), J, B, J, J, ARD_ACT_NONE, s));
        ARD_TRY(l2_normalize(h->ws_proj.as<float>(), a->audio_embed, B, J, s));
    }
    if (need_tscam) {
        if (a->fine_grained_embedding) ARD_TRY(fine_grained(normed, a->fine_grained_embedding, B, NF, s));
        if (a->framewise_output || a->clipwise_output) {
            if (!h->tscam_w.p) return set_error(ARD_ERR_STATE, "tscam_conv weights were never set");
            const int ldy = 528;
            ARD_TRY(h->ws_tscam_y.ensure((size_t)B * 32 * ldy * 4));
            if (fp32) {
                ARD_TRY(tscam_gemm_fp32(h, normed, h->ws_tscam_y.as<float>(), ldy, B, s));
            } else {
                ARD_TRY(h->ws_tscam_a.ensure((size_t)B * 32 * NF * 6 * 2));
                ARD_TRY(tscam_im2col(normed, h->ws_tscam_a.as<__nv_bfloat16>(), B, NF, s));
                GemmArgs g;
                g.A = h->ws_tscam_a.as<__nv_bfloat16>(); g.lda = 6LL * NF; g.W = h->tscam_w.as<__nv_bfloat16>(); g.ldw = 6LL * NF;
                g.out = h->ws_tscam_y.as<float>(); g.ldo = ldy; g.M = B * 32; g.N = ARD_CLASS_NUM; g.K = 6 * NF; g.bias = h->tscam_b.as<float>();
                ARD_TRY(gemm_bf16(g, h->num_sms, s));
            }
            ARD_TRY(tscam_finish(h->ws_tscam_y.as<float>(), ldy, a->framewise_output, a->clipwise_output, B, ARD_CLASS_NUM, s));
        }
    }
    return 0;
}

}  // namespace ard

// ================================================================================================== C ABI
extern "C" {

const char* ard_last_error(void) { return g_err; }
int ard_version(void) { return 100; }

int ard_create(const ard_config* cfg, ard_handle** out) {
    if (!cfg || !out) return set_error(ARD_ERR_SHAPE, "null argument");
    if (cfg->embed_dim != 96 && cfg->embed_dim != 128)
        return set_error(ARD_ERR_SHAPE, "Import Model for embed_dim=%d not found (tiny=96, base=128)", cfg->embed_dim);   // htsat.py:1044-1045
    ard_handle* h = new ard_handle();
    h->cfg = *cfg;
    h->layers.resize(4);
    for (int l = 0; l < 4; ++l) {
        if (cfg->depths[l] <= 0 || cfg->num_heads[l] <= 0) { delete h; return set_error(ARD_ERR_SHAPE, "bad depth/heads for layer %d", l); }
        h->layers[l].blocks.resize(cfg->depths[l]);
    }
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        delete h;
        return set_error(ARD_ERR_CUDA, "no CUDA device: libard_b200 has no CPU fallback");
    }
    h->num_sms = sms;
    if (const char* e = getenv("ARD_FUSED_FFN")) h->use_fused_ffn = atoi(e) != 0;
    if (const char* e = getenv("ARD_FUSED_FFN_WIDE")) h->use_fused_ffn_wide = atoi(e);
    if (const char* e = getenv("ARD_GRAPHS")) h->use_graphs = atoi(e);
    if (const char* e = getenv("ARD_LN_QKV")) h->use_ln_qkv = atoi(e) != 0;
    if (const char* e = getenv("ARD_ATTN_BLOCK")) h->use_attn_block = atoi(e) != 0;
    if (const char* e = getenv("ARD_DUAL_GEMM")) h->use_dual_gemm = atoi(e);
    *out = h;
    return 0;
}

int ard_destroy(ard_handle* h) {
    delete h;
    return 0;
}

int ard_set_weight(ard_handle* h, const char* key, const float* data, long long numel) {
    if (!h || !key || !data || numel <= 0) return set_error(ARD_ERR_SHAPE, "ard_set_weight: bad argument");
    h->host[std::string(key)] = std::vector<float>(data, data + numel);
    h->finalized = false;
    ++h->graph_epoch;
    return 0;
}

int ard_finalize_weights(ard_handle* h, void* stream) {
    if (!h) return set_error(ARD_ERR_SHAPE, "null handle");
    return finalize(h, (cudaStream_t)stream);
}

int ard_set_block_residual(ard_handle* h, int layer, int block, const float* mean, const float* basis, int K, int D) {
    if (!h) return set_error(ARD_ERR_SHAPE, "null handle");
    if (layer < 0 || layer >= h->nlayers) return set_error(ARD_ERR_SHAPE, "Layer index %d out of range for model with %d layers", layer, h->nlayers);  // src/residual.py:194-195
    if (block < 0 || block >= h->cfg.depths[layer]) return set_error(ARD_ERR_SHAPE, "block index %d out of range", block);
    const int C = C_of(h, layer);
    if (D != C || K <= 0 || K > D) return set_error(ARD_ERR_SHAPE, "ResiDual basis [%d,%d] does not match layer width %d", K, D, C);
    BlockW& bw = h->layers[layer].blocks[block];
    ++h->graph_epoch;
    bw.K = K;
    bw.h_mean.assign(mean, mean + D);
    bw.h_basis.assign(basis, basis + (size_t)K * D);
    bw.bwd_ready = false;
    ARD_TRY(upload(bw.res_basis, basis, (size_t)K * D * 4));
    ARD_TRY(bw.res_M.ensure((size_t)C * C * 4));
    ARD_TRY(bw.proj_w_fold.ensure((size_t)C * C * 2));
    ARD_TRY(bw.proj_w_fold_f32.ensure((size_t)C * C * 4));
    ARD_TRY(bw.proj_b_fold.ensure((size_t)C * 4));
    char key[96];
    snprintf(key, sizeof(key), "layers.%d.blocks.%d.attn.proj.bias", layer, block);
    auto it = h->host.find(key);
    if (it == h->host.end()) return set_error(ARD_ERR_STATE, "set weights before injecting ResiDual ('%s' missing)", key);
    std::vector<float> dm(C);
    for (int i = 0; i < C; ++i) dm[i] = it->second[i] - mean[i];
    ARD_TRY(upload_f32(bw.res_dmean, dm));
    bw.has_res = true;
    bw.lambda_set = false;
    if (bw.lam.p) { cudaFree(bw.lam.p); bw.lam.p = nullptr; bw.lam.bytes = 0; }
    return 0;
}

int ard_clear_block_residual(ard_handle* h, int layer, int block) {
    if (!h || layer < 0 || layer >= h->nlayers || block < 0 || block >= h->cfg.depths[layer]) return set_error(ARD_ERR_SHAPE, "bad block index");
    h->layers[layer].blocks[block].has_res = false;
    ++h->graph_epoch;
    return 0;
}

// what a block needs after its fold changed: the padded copies of the attention-block kernel, and lambda for the backward
static int after_fold(ard_handle* h, int layer, BlockW& bw, const float* lambda_dev, cudaStream_t s) {
    const int C = C_of(h, layer);
    if (bw.ab.ready)
        ARD_TRY(attn_block_pad_proj(bw.proj_w_fold.as<__nv_bfloat16>(), bw.proj_b_fold.as<float>(), bw.ab.bv.as<float>(), bw.ab.wp_fold.as<__nv_bfloat16>(),
                                    bw.ab.bp_fold.as<float>(), C, h->cfg.num_heads[layer], s));
    // keep a (zero-padded) copy of lambda for the backward: gsc = gcoef * lambda
    const int Kp = (bw.K + 15) & ~15;
    ARD_TRY(bw.lam.ensure((size_t)Kp * 4));
    ARD_CUDA(cudaMemsetAsync(bw.lam.p, 0, (size_t)Kp * 4, s));
    ARD_CUDA(cudaMemcpyAsync(bw.lam.p, lambda_dev, (size_t)bw.K * 4, cudaMemcpyDeviceToDevice, s));
    bw.lambda_set = true;
    return 0;
}

int ard_set_block_lambda(ard_handle* h, int layer, int block, const float* lambda_dev, void* stream) {
    if (!h || layer < 0 || layer >= h->nlayers || block < 0 || block >= h->cfg.depths[layer]) return set_error(ARD_ERR_SHAPE, "bad block index");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    BlockW& bw = h->layers[layer].blocks[block];
    if (!bw.has_res) return set_error(ARD_ERR_STATE, "block (%d,%d) has no ResiDual injected", layer, block);
    const int C = C_of(h, layer);
    g_launches = 0;
    ARD_TRY(residual_fold(bw.proj_w_f32.as<float>(), bw.res_dmean.as<float>(), bw.res_basis.as<float>(), lambda_dev, C, bw.K,
                          bw.res_M.as<float>(), bw.proj_w_fold.as<__nv_bfloat16>(), bw.proj_b_fold.as<float>(), (cudaStream_t)stream,
                          bw.proj_w_fold_f32.as<float>()));
    return after_fold(h, layer, bw, lambda_dev, (cudaStream_t)stream);
}

// The reference builds ONE ResiDual per layer and shares it between the layer's blocks (src/residual.py:170-186), so
// M = B^T diag(lambda) B is a per-layer matrix: it is formed once and the folds of all patched blocks of the layer run as one
// batched launch each (3 launches per layer instead of 3 per block; the training step re-folds every layer every step).
int ard_set_layer_lambda(ard_handle* h, int layer, const float* lambda_dev, void* stream) {
    if (!h || layer < 0 || layer >= h->nlayers) return set_error(ARD_ERR_SHAPE, "bad layer index");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    const int C = C_of(h, layer);
    cudaStream_t s = (cudaStream_t)stream;
    std::vector<BlockW*> pb;
    for (BlockW& bw : h->layers[layer].blocks)
        if (bw.has_res) pb.push_back(&bw);
    if (pb.empty()) return set_error(ARD_ERR_STATE, "layer %d has no ResiDual injected", layer);
    for (BlockW* bw : pb)   // the caller states the blocks share one ResiDual: same basis and mean (host copies kept by ard_set_block_residual)
        if (bw->K != pb[0]->K || bw->h_basis != pb[0]->h_basis || bw->h_mean != pb[0]->h_mean)
            return set_error(ARD_ERR_STATE, "layer %d: its blocks carry different ResiDual bases; use ard_set_block_lambda per block", layer);
    g_launches = 0;
    for (size_t i0 = 0; i0 < pb.size(); i0 += 8) {
        const int nb = (int)std::min<size_t>(8, pb.size() - i0);
        const float *pw[8], *dm[8];
        __nv_bfloat16* wo[8];
        float *bo[8], *wf[8];
        for (int z = 0; z < nb; ++z) {
            BlockW& bw = *pb[i0 + z];
            pw[z] = bw.proj_w_f32.as<float>(); dm[z] = bw.res_dmean.as<float>(); wo[z] = bw.proj_w_fold.as<__nv_bfloat16>();
            bo[z] = bw.proj_b_fold.as<float>(); wf[z] = bw.proj_w_fold_f32.as<float>();
        }
        ARD_TRY(residual_fold_batch(pw, dm, pb[0]->res_basis.as<float>(), lambda_dev, C, pb[0]->K, pb[0]->res_M.as<float>(), wo, bo, wf, nb, s));
    }
    for (BlockW* bw : pb) ARD_TRY(after_fold(h, layer, *bw, lambda_dev, s));
    return 0;
}

// Inference forward with only the pooled outputs requested: replayed from a CUDA graph keyed by (input pointer, batch,
// quantize, audio_embed wanted). First use runs kernel by kernel (allocates workspaces, folds lambdas), second use captures,
// later uses replay. The graph writes handle-owned output buffers; two small device copies hand the result to the caller, so
// freshly allocated output tensors do not defeat the cache. Anything that moves a device buffer or changes the schedule
// (weights, ResiDual injection, a larger workspace) bumps an epoch and the entry is re-captured.
static int forward_graphed(ard_handle* h, const ard_forward_args* args, cudaStream_t s, bool* handled) {
    *handled = false;
    const bool eligible = h->use_graphs && h->finalized && !g_prof_on && !args->save_for_backward && args->precision == 0 && args->B > 0 && args->embedding &&
                          !args->framewise_output && !args->clipwise_output && !args->fine_grained_embedding &&
                          !args->layers_residuals[0] && !args->layers_residuals[1] && !args->layers_residuals[2] && !args->layers_residuals[3] &&
                          !args->layers_attention[0] && !args->layers_attention[1] && !args->layers_attention[2] && !args->layers_attention[3] &&
                          !args->head_outputs[0] && !args->head_outputs[1] && !args->head_outputs[2] && !args->head_outputs[3];
    if (!eligible) return 0;
    const void* src = h->cfg.enable_fusion ? (const void*)args->mel_fusion : (const void*)args->waveform;
    if (!src) return 0;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return 0;   // the caller is capturing: stay out of it
    const int NF = C_of(h, h->nlayers - 1), J = h->cfg.joint_dim, B = args->B;
    ard_handle::GraphKey key{src, B, args->quantize, args->audio_embed != nullptr};
    auto it = h->graphs.find(key);
    const bool fresh = it != h->graphs.end() && it->second.epoch == h->graph_epoch && it->second.aepoch == alloc_epoch();
    if (!fresh) {
        // first sighting (or stale): run eagerly, make sure everything a capture must not allocate exists, remember the key
        if (it != h->graphs.end() && it->second.exec) { cudaGraphExecDestroy(it->second.exec); it->second.exec = nullptr; }
        if (h->graphs.size() >= 32 && it == h->graphs.end()) {   // bounded cache: drop the least recently used entry
            auto lru = h->graphs.begin();
            for (auto jt = h->graphs.begin(); jt != h->graphs.end(); ++jt)
                if (jt->second.last_use < lru->second.last_use) lru = jt;
            if (lru->second.exec) cudaGraphExecDestroy(lru->second.exec);
            h->graphs.erase(lru);
        }
        const int rc = encoder_forward(h, args, s);
        *handled = true;
        if (rc) return rc;
        ARD_TRY(h->g_emb.ensure((size_t)B * NF * 4));
        ARD_TRY(h->g_ae.ensure((size_t)B * J * 4));
        ard_handle::GraphEntry e;
        e.epoch = h->graph_epoch; e.aepoch = alloc_epoch(); e.last_use = ++h->graph_clock;
        h->graphs[key] = e;
        return 0;
    }
    ard_handle::GraphEntry& e = it->second;
    e.last_use = ++h->graph_clock;
    if (!e.exec) {
        ard_forward_args a2 = *args;
        a2.embedding = h->g_emb.as<float>();
        if (args->audio_embed) a2.audio_embed = h->g_ae.as<float>();
        const int before = g_launches;
        if (!h->cap_stream && cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError(); h->cap_stream = nullptr; h->use_graphs = 0; return 0;
        }
        if (cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); h->use_graphs = 0; return 0; }
        const int rc = encoder_forward(h, &a2, h->cap_stream);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &graph);
        const int captured = g_launches - before;
        g_launches = before; g_launch_total -= captured;      // nothing ran yet
        if (rc || ce != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            h->graphs.erase(it);
            return 0;                                          // fall back to the eager path
        }
        cudaGraphExec_t exec = nullptr;
        const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess || !exec) { cudaGetLastError(); h->graphs.erase(it); return 0; }
        e.exec = exec;
        e.launches = captured;
    }
    ARD_CUDA(cudaGraphLaunch(e.exec, s));
    count_launch(e.launches);
    ARD_CUDA(cudaMemcpyAsync(args->embedding, h->g_emb.p, (size_t)B * NF * 4, cudaMemcpyDeviceToDevice, s));
    if (args->audio_embed) ARD_CUDA(cudaMemcpyAsync(args->audio_embed, h->g_ae.p, (size_t)B * J * 4, cudaMemcpyDeviceToDevice, s));
    h->tape_B = 0;
    *handled = true;
    return 0;
}

int ard_encoder_forward(ard_handle* h, const ard_forward_args* args, void* stream) {
    if (!h || !args) return set_error(ARD_ERR_SHAPE, "null argument");
    g_launches = 0;
    bool handled = false;
    int rc = forward_graphed(h, args, (cudaStream_t)stream, &handled);
    if (!handled && rc == 0) rc = encoder_forward(h, args, (cudaStream_t)stream);
    h->last_launches = g_launches;
    return rc;
}

int ard_block_forward(ard_handle* h, int layer, int block, const float* x_in, int B, float* x_out, float* attn, float* residual_x,
                      void* stream) {
    if (!h || !x_in || !x_out) return set_error(ARD_ERR_SHAPE, "null argument");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    if (layer < 0 || layer >= h->nlayers || block < 0 || block >= h->cfg.depths[layer]) return set_error(ARD_ERR_SHAPE, "bad block index");
    if (B <= 0) return set_error(ARD_ERR_SHAPE, "batch must be positive");
    cudaStream_t s = (cudaStream_t)stream;
    g_launches = 0;
    ARD_TRY(ensure_workspace(h, B));
    const int C = C_of(h, layer), T = R_of(layer) * R_of(layer);
    const size_t bytes = (size_t)B * T * C * 4;
    float* X = h->ws_x.as<float>();
    float* Y = h->ws_y.as<float>();
    ARD_CUDA(cudaMemcpyAsync(X, x_in, bytes, cudaMemcpyDeviceToDevice, s));
    const BlockIO io{X, Y, Y, X, h->ws_qkv.as<__nv_bfloat16>(), h->ws_ao.as<__nv_bfloat16>(), false};
    ARD_TRY(run_block(h, layer, block, B, io, attn, 1.0f, 0, residual_x, T, nullptr, s));
    ARD_CUDA(cudaMemcpyAsync(x_out, X, bytes, cudaMemcpyDeviceToDevice, s));
    h->last_launches = g_launches;
    return 0;
}

int ard_attention_block(ard_handle* h, int layer, int block, const float* x_in, int B, float* x_out, void* stream) {
    if (!h || !x_in || !x_out) return set_error(ARD_ERR_SHAPE, "null argument");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    if (layer < 0 || layer >= h->nlayers || block < 0 || block >= h->cfg.depths[layer]) return set_error(ARD_ERR_SHAPE, "bad block index");
    if (B <= 0) return set_error(ARD_ERR_SHAPE, "batch must be positive");
    BlockW& bw = h->layers[layer].blocks[block];
    if (!bw.ab.ready) return set_error(ARD_ERR_NOTIMPL, "the window-resident attention block kernel covers the 96-channel stage (layer 0 of HTSAT-tiny)");
    cudaStream_t s = (cudaStream_t)stream;
    g_launches = 0;
    ARD_TRY(ensure_fold(h, layer, block, s));
    const int R = R_of(layer);
    const int rc = attn_block_96(x_in, x_out, bw.ab, (bw.has_res ? bw.ab.wp_fold : bw.ab.wp_plain).as<__nv_bfloat16>(),
                                 (bw.has_res ? bw.ab.bp_fold : bw.ab.bp_plain).as<float>(), bw.ln1_g.as<float>(), bw.ln1_b.as<float>(), B, R,
                                 (block % 2 == 0) ? 0 : 4, h->num_sms, s);
    h->last_launches = g_launches;
    return rc;
}

int ard_encoder_backward_outputs(ard_handle* h, const ard_backward_args* args, const ard_output_grads* outs, void* stream) {
    if (!h || !args) return set_error(ARD_ERR_SHAPE, "null argument");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    g_launches = 0;
    const int rc = encoder_backward(h, args, outs, (cudaStream_t)stream);
    h->last_launches = g_launches;
    return rc;
}

int ard_encoder_backward(ard_handle* h, const ard_backward_args* args, void* stream) {
    return ard_encoder_backward_outputs(h, args, nullptr, stream);
}

int ard_tail_backward(ard_handle* h, const float* y, int ldy, const float* grad_framewise, const float* grad_clipwise, const float* grad_fine,
                      const float* grad_embedding, int B, int precision, float* grad_normed, void* stream) {
    if (!h || !grad_normed) return set_error(ARD_ERR_SHAPE, "null argument");
    if (!h->finalized) return set_error(ARD_ERR_STATE, "ard_finalize_weights has not been called");
    if (B <= 0 || (precision != 0 && precision != 1)) return set_error(ARD_ERR_SHAPE, "ard_tail_backward: B = %d, precision = %d", B, precision);
    if ((grad_framewise || grad_clipwise) && (!y || ldy < ARD_CLASS_NUM))
        return set_error(ARD_ERR_SHAPE, "ard_tail_backward: the framewise / clipwise terms need y [B*32, ldy >= 527]");
    g_launches = 0;
    const int rc = tail_backward(h, y, ldy, grad_framewise, grad_clipwise, grad_fine, grad_embedding, B, precision == 1, grad_normed,
                                 (cudaStream_t)stream);
    h->last_launches = g_launches;
    return rc;
}

long long ard_tape_generation(const ard_handle* h) { return h && h->tape_B > 0 ? h->tape_gen : 0; }

long long ard_workspace_bytes(const ard_handle* h) {
    if (!h) return 0;
    const DevBuf* bufs[] = {&h->ws_logmel, &h->ws_x, &h->ws_y, &h->ws_xn, &h->ws_ao, &h->ws_qkv, &h->ws_h, &h->ws_normed,
                            &h->ws_hid, &h->ws_proj, &h->ws_tscam_a, &h->ws_tscam_y, &h->tape, &h->bw_g, &h->bw_gs, &h->bw_t,
                            &h->bw_dh, &h->bw_gb, &h->bw_coef, &h->bw_gcoef, &h->bw_gsc, &h->bw_small, &h->bw_g3,
                            &h->bw_tail_dy, &h->bw_tail_da};
    long long t = 0;
    for (const DevBuf* b : bufs) t += (long long)b->bytes;
    return t;
}
int ard_last_launch_count(const ard_handle* h) { return h ? h->last_launches : 0; }
int ard_launch_counter_reset(void) { g_launch_total = 0; return 0; }
long long ard_launch_counter_read(void) { return g_launch_total; }

// ---------------------------------------------------------------- op-level entry points
int ard_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_is_bf16, int M, int N,
                  int K, const float* bias, int act, const float* resid1, long long ldr1, const float* resid2, long long ldr2,
                  void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    GemmArgs g;
    g.A = (const __nv_bfloat16*)A; g.lda = lda; g.W = (const __nv_bfloat16*)W; g.ldw = ldw; g.out = out; g.ldo = ldo; g.out_bf16 = out_is_bf16;
    g.M = M; g.N = N; g.K = K; g.bias = bias; g.act = act; g.resid1 = resid1; g.ldr1 = ldr1; g.resid2 = resid2; g.ldr2 = ldr2;
    if (act == ARD_ACT_GELU_F16) { g.act = ARD_ACT_GELU; g.out_f16 = 1; }
    return gemm_bf16(g, sms, (cudaStream_t)stream);
}

int ard_gemm_dual(int mode, const void* A1, long long lda1, const void* W1, long long ldw1, const void* A2, long long lda2, const void* W2,
                  long long ldw2, void* out, long long ldo, int M, int N, int K, const float* vec1, const float* vec2, float* dlam, int Kvalid,
                  void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    if (mode != 0 && mode != 1) return set_error(ARD_ERR_SHAPE, "ard_gemm_dual: mode must be 0 (gelu backward) or 1 (lambda gradient)");
    DualArgs d;
    d.A1 = (const __nv_bfloat16*)A1; d.lda1 = lda1; d.W1 = (const __nv_bfloat16*)W1; d.ldw1 = ldw1;
    d.A2 = (const __nv_bfloat16*)A2; d.lda2 = lda2; d.W2 = (const __nv_bfloat16*)W2; d.ldw2 = ldw2;
    d.out = (__nv_bfloat16*)out; d.ldo = ldo; d.M = M; d.N = N; d.K = K; d.vec1 = vec1; d.vec2 = vec2; d.dlam = dlam; d.Kvalid = Kvalid;
    return mode == 0 ? gemm_dual_gelu_bwd(d, sms, (cudaStream_t)stream) : gemm_dual_lambda(d, sms, (cudaStream_t)stream);
}

int ard_gemm_f16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_is_bf16, int M, int N,
                 int K, const float* bias, int act, const float* resid1, long long ldr1, const float* resid2, long long ldr2,
                 void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    GemmArgs g;
    g.A = (const __nv_bfloat16*)A; g.lda = lda; g.W = (const __nv_bfloat16*)W; g.ldw = ldw; g.out = out; g.ldo = ldo; g.out_bf16 = out_is_bf16;
    g.M = M; g.N = N; g.K = K; g.bias = bias; g.act = act; g.resid1 = resid1; g.ldr1 = ldr1; g.resid2 = resid2; g.ldr2 = ldr2;
    g.ab_f16 = 1;
    return gemm_bf16(g, sms, (cudaStream_t)stream);
}

int ard_ffn_fused_96(const float* x, const float* resid2, float* out, long long M, const float* gamma, const float* beta, const void* w1_bf16,
                     const float* b1, const void* w2_f16, const float* b2, void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    return ffn_fused_96(x, resid2, out, M, gamma, beta, (const __nv_bfloat16*)w1_bf16, b1, (const __half*)w2_f16, b2, sms,
                        (cudaStream_t)stream);
}

int ard_ffn_fused_wide(const float* x, const float* resid2, float* out, long long M, int C, const float* gamma, const float* beta,
                       const void* w1_bf16, const float* b1_half, const void* w2_f16, const float* b2, void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    return ffn_fused_wide(x, resid2, out, M, C, gamma, beta, (const __nv_bfloat16*)w1_bf16, b1_half, (const __half*)w2_f16, b2, sms,
                          (cudaStream_t)stream);
}

int ard_ln_qkv_96(const float* x, const float* gamma, const float* beta, const void* w_bf16, const float* bias, void* qkv_bf16, long long M,
                  void* stream) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(ARD_ERR_CUDA, "no CUDA device");
    return ln_qkv_96(x, gamma, beta, (const __nv_bfloat16*)w_bf16, bias, (__nv_bfloat16*)qkv_bf16, M, sms, (cudaStream_t)stream);
}

int ard_layernorm_bf16(const float* x, const float* gamma, const float* beta, void* out_bf16, long long rows, int C, void* stream) {
    return layernorm_bf16(x, gamma, beta, (__nv_bfloat16*)out_bf16, rows, C, (cudaStream_t)stream);
}

int ard_window_attention(const void* qkv_bf16, void* out_bf16, const float* bias_table, float* attn, float attn_scale, int accumulate,
                         int B, int H, int W, int C, int nH, int shift, void* stream) {
    AttnArgs a;
    a.qkv = (const __nv_bfloat16*)qkv_bf16; a.out = (__nv_bfloat16*)out_bf16; a.bias_table = bias_table; a.attn_mean = attn;
    a.attn_scale = attn_scale; a.attn_accumulate = accumulate; a.B = B; a.H = H; a.W = W; a.C = C; a.nH = nH; a.shift = shift;
    return window_attention(a, (cudaStream_t)stream);
}

int ard_window_attention_bwd(const void* qkv_bf16, const void* dout_bf16, void* dqkv_bf16, const float* bias_table, int B, int H, int W, int C,
                             int nH, int shift, void* stream) {
    AttnArgs a;
    a.qkv = (const __nv_bfloat16*)qkv_bf16; a.bias_table = bias_table; a.B = B; a.H = H; a.W = W; a.C = C; a.nH = nH; a.shift = shift;
    return window_attention_bwd(a, (const __nv_bfloat16*)dout_bf16, (__nv_bfloat16*)dqkv_bf16, (cudaStream_t)stream);
}

int ard_window_attention_f32_bwd(const float* qkv_f32, const float* dout_f32, float* dqkv_f32, const float* bias_table, int B, int H, int W,
                                 int C, int nH, int shift, void* stream) {
    if (!qkv_f32 || !dout_f32 || !dqkv_f32 || !bias_table) return set_error(ARD_ERR_SHAPE, "ard_window_attention_f32_bwd: null argument");
    if (H != W) return set_error(ARD_ERR_SHAPE, "ard_window_attention_f32_bwd: square token grids only (H=%d W=%d)", H, W);
    return window_attention_f32_bwd(qkv_f32, dout_f32, dqkv_f32, bias_table, B, H, C, nH, shift, (cudaStream_t)stream);
}

int ard_window_attention_bwd_pgrad(const void* qkv_bf16, const void* dout_bf16, const float* pgrad, float pscale, void* dqkv_bf16,
                                   const float* bias_table, int B, int H, int W, int C, int nH, int shift, void* stream) {
    if (!pgrad) return set_error(ARD_ERR_SHAPE, "ard_window_attention_bwd_pgrad: null probability gradient");
    AttnArgs a;
    a.qkv = (const __nv_bfloat16*)qkv_bf16; a.bias_table = bias_table; a.B = B; a.H = H; a.W = W; a.C = C; a.nH = nH; a.shift = shift;
    return window_attention_bwd(a, (const __nv_bfloat16*)dout_bf16, (__nv_bfloat16*)dqkv_bf16, (cudaStream_t)stream, pgrad, pscale);
}

int ard_window_attention_f32_bwd_pgrad(const float* qkv_f32, const float* dout_f32, const float* pgrad, float pscale, float* dqkv_f32,
                                       const float* bias_table, int B, int H, int W, int C, int nH, int shift, void* stream) {
    if (!qkv_f32 || !dout_f32 || !pgrad || !dqkv_f32 || !bias_table) return set_error(ARD_ERR_SHAPE, "ard_window_attention_f32_bwd_pgrad: null argument");
    if (H != W) return set_error(ARD_ERR_SHAPE, "ard_window_attention_f32_bwd_pgrad: square token grids only (H=%d W=%d)", H, W);
    return window_attention_f32_bwd(qkv_f32, dout_f32, dqkv_f32, bias_table, B, H, C, nH, shift, (cudaStream_t)stream, pgrad, pscale);
}

int ard_layernorm_bwd(const float* x, const float* grad_out, const float* gamma, const float* add, float* grad_in, long long rows, int C,
                      void* stream) {
    return layernorm_bwd(x, grad_out, gamma, add, grad_in, rows, C, (cudaStream_t)stream, 1.0f, nullptr);
}

int ard_f32_to_bf16(const float* in, void* out_bf16, long long n, float scale, void* stream) {
    return f32_to_bf16(in, (__nv_bfloat16*)out_bf16, n, scale, (cudaStream_t)stream);
}

int ard_quantize_waveform(const float* in, float* out, long long n, void* stream) { return quantize_waveform(in, out, n, (cudaStream_t)stream); }

int ard_logmel(ard_handle* h, const float* wave, int B, int n_samples, int apply_bn, int quantize, float* out, void* stream) {
    if (!h || !h->finalized) return set_error(ARD_ERR_STATE, "handle not finalised");
    if (!h->window.p) return set_error(ARD_ERR_STATE, "front-end weights (spectrogram_extractor / logmel_extractor) were never set");
    MelBands mb{h->melw.as<float>(), h->mstart.as<int>(), h->mlen.as<int>(), h->band_max};
    return stft_logmel(wave, B, n_samples, h->window.as<float>(), h->twiddle.as<float2>(), mb, apply_bn ? h->bn_scale.as<float>() : nullptr,
                       apply_bn ? h->bn_shift.as<float>() : nullptr, out, 0, 1, quantize, (cudaStream_t)stream);
}

int ard_patch_embed(ard_handle* h, const float* logmel, int B, float* out, void* stream) {
    if (!h || !h->finalized) return set_error(ARD_ERR_STATE, "handle not finalised");
    if (!logmel || !out || B <= 0) return set_error(ARD_ERR_SHAPE, "ard_patch_embed: bad argument");
    return patch_embed_ln(logmel, (long long)ARD_FRAMES * 64, ARD_FRAMES, h->bn_scale.as<float>(), h->bn_shift.as<float>(), h->pe_w.as<float>(),
                          h->pe_b.as<float>(), h->pe_g.as<float>(), h->pe_beta.as<float>(), out, B, h->cfg.embed_dim, (cudaStream_t)stream);
}

int ard_fusion_mel(ard_handle* h, const float* wave, int B, int n_samples, int quantize, float* out, void* stream) {
    if (!h || !h->finalized) return set_error(ARD_ERR_STATE, "handle not finalised");
    if (!h->f_window.p) return set_error(ARD_ERR_STATE, "fusion featuriser tensors (fusion_featuriser.melW / .window) were never set");
    MelBands mb{h->f_melw.as<float>(), h->f_mstart.as<int>(), h->f_mlen.as<int>(), h->f_band_max};
    const int frames = n_samples / 480 + 1;
    return stft_logmel(wave, B, n_samples, h->f_window.as<float>(), h->twiddle.as<float2>(), mb, nullptr, nullptr, out,
                       4LL * frames * 64, 4, quantize, (cudaStream_t)stream);
}

int ard_stats_accumulate(const float* x, long long rows, int D, double* sum, double* sumsq, void* stream) {
    return stats_accumulate(x, rows, D, D, sum, sumsq, (cudaStream_t)stream);
}

int ard_stats_accumulate_strided(const float* x, long long rows, long long ldx, int D, double* sum, double* sumsq, void* stream) {
    return stats_accumulate(x, rows, ldx, D, sum, sumsq, (cudaStream_t)stream);
}

int ard_profile_enable(int on) {
    g_prof_on = on != 0;
    return 0;
}

int ard_profile_read(double* ms, double* flops, double* bytes, int* launches, int nclass) {
    if (nclass < PROF_NCLASS) return set_error(ARD_ERR_SHAPE, "ard_profile_read: need %d classes", (int)PROF_NCLASS);
    for (int i = 0; i < nclass; ++i) { ms[i] = 0; flops[i] = 0; bytes[i] = 0; launches[i] = 0; }
    ARD_CUDA(cudaDeviceSynchronize());
    for (ProfRec& r : g_prof) {
        float t = 0.f;
        cudaEventElapsedTime(&t, r.a, r.b);
        ms[r.cls] += t; flops[r.cls] += r.flops; bytes[r.cls] += r.bytes; launches[r.cls] += 1;
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_prof.clear();
    return 0;
}

}  // extern "C"
