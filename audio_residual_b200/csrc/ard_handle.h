// Handle layout shared by ard_api.cu (forward schedule, C ABI), ard_train.cu (tape layout + backward schedule) and
// fp32_mode.cu (fp32-grade forward).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "ard_internal.h"

namespace ard {

// ------------------------------------------------------------------------------------------------ device buffers
// bumped whenever a device buffer is (re)allocated: captured CUDA graphs hold raw pointers and are stale afterwards
inline unsigned long long& alloc_epoch() {
    static unsigned long long e = 0;
    return e;
}

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    int ensure(size_t n) {
        if (n <= bytes) return 0;
        ++alloc_epoch();
        if (p) { cudaFree(p); p = nullptr; bytes = 0; }
        cudaError_t e = cudaMalloc(&p, n);
        if (e != cudaSuccess) { p = nullptr; return set_error(ARD_ERR_CUDA, "cudaMalloc(%zu): %s", n, cudaGetErrorString(e)); }
        bytes = n;
        return 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// padded per-head q/k/v weights of the window-resident attention block kernel (attn_block.cu), 96-channel stage
struct AttnBlockW {
    DevBuf wqk, bq, wv, bv, table, wp_plain, wp_fold, bp_plain, bp_fold;   // [256,96] bf16, [128] f32, [128,96] bf16, [96] f32 (un-padded v bias),
                                                                           // [4,15,24] f32, 2 x [96,128] bf16, 2 x [96] f32 (bias + Wp' bv)
    bool ready = false;
};

struct BlockW {
    DevBuf ln1_g, ln1_b, ln2_g, ln2_b;
    DevBuf qkv_w, qkv_b, proj_w, proj_b, proj_w_f32, fc1_w, fc1_b, fc1_b_half, fc2_w, fc2_b, rpb;
    // ResiDual (src/residual.py:14-42) injected after this block's attention
    bool has_res = false, lambda_set = false;
    int K = 0;
    std::vector<float> h_mean, h_basis;
    DevBuf res_basis, res_dmean, res_M, proj_w_fold, proj_w_fold_f32, proj_b_fold, lam_ones;
    AttnBlockW ab;
    // training (ard_train.cu): current lambda (padded to Kp), transposed / folded weights for the dgrad GEMMs, built lazily
    int Kp = 0;
    bool bwd_ready = false;
    DevBuf lam, fc1_wT, fc2_wT, qkv_wT, proj_wT, res_wc, res_wcT, res_basis_bf16, res_c0;
    // activations saved by a save_for_backward forward (views into ard_handle::tape, the block's BlockIO / Fp32BlockIO in that
    // forward); qkv / ao are bf16 on a bf16 tape (t_qkv, t_ao) and fp32 on an fp32-grade tape (t_qkvf, t_aof), the other pair is null
    float *t_s = nullptr, *t_x1 = nullptr, *t_x3 = nullptr, *t_out = nullptr;
    __nv_bfloat16 *t_qkv = nullptr, *t_ao = nullptr;
    float *t_qkvf = nullptr, *t_aof = nullptr;
};
struct LayerW {
    std::vector<BlockW> blocks;
    DevBuf mg_g, mg_b, mg_w, mg_wT;
};

// fp32-grade mode (fp32_mode.cu). Split weights [W_hi | W_lo | W_hi] ([N, 3K] bf16) of the forward GEMMs and, built on the
// first fp32-grade backward, of the backward's dgrad GEMMs; all rebuilt when ard_handle::graph_epoch moves.
struct Fp32BlockW {
    DevBuf qkv3, proj3, fc13, fc23;
    DevBuf fc1T3, fc2T3, qkvT3, projT3;                // [C, 3*4C], [4C, 3C], [C, 3*3C] (q rows pre-scaled), [C, 3C]
    DevBuf wc3, wcT3, basis3;                          // ResiDual: Wc = B Wp [Kp, 3C], Wc^T [C, 3Kp], basis padded to Kp [Kp, 3C]
};
struct Fp32Weights {
    unsigned long long epoch = ~0ULL;            // ard_handle::graph_epoch the split weights were built at (weights / ResiDual changes bump it)
    unsigned long long bwd_epoch = ~0ULL;        // the same for the backward set (built by the first fp32-grade backward after a change)
    unsigned long long tscam_epoch = ~0ULL;      // the same for tscamT3 (built by the first fp32-grade tail backward after a change)
    std::vector<std::vector<Fp32BlockW>> blocks;
    std::vector<DevBuf> merge3, mergeT3;         // PatchMerging reduction [2C, 3*4C] and its transpose [4C, 3*2C] (backward, lazily)
    DevBuf tscam3, tscamT3, scratch;                   // tscam_conv [527, 3*6C] and, for the tail backward, its transpose [6C, 3*528]
    DevBuf fold3;                                // folded projection of the block being run: depends on the current lambda, re-split per call
    DevBuf qkvf, aof, s3;                        // workspace: fp32 [M,4C] (qkv / FFN hidden), fp32 [M,C], split operands [M,12C] bf16
};

}  // namespace ard

struct ard_handle {
    using DevBuf = ard::DevBuf;
    using LayerW = ard::LayerW;
    using Fp32Weights = ard::Fp32Weights;
    ard_config cfg;
    int nlayers = 4;
    int num_sms = 148;
    bool finalized = false;
    std::map<std::string, std::vector<float>> host;   // raw state_dict tensors (fp32)
    // front end
    DevBuf window, twiddle, melw, mstart, mlen, bn_scale, bn_shift;
    int band_max = 0;
    DevBuf f_window, f_melw, f_mstart, f_mlen;   // fusion featuriser (get_mel, data.py:363-399): htk filters, periodic hann
    int f_band_max = 0;
    DevBuf pe_w, pe_b, pe_g, pe_beta;
    std::vector<LayerW> layers;
    DevBuf norm_g, norm_b, tscam_w, tscam_b, p0_w, p0_b, p2_w, p2_b;
    // workspace
    DevBuf ws_logmel, ws_x, ws_y, ws_xn, ws_ao, ws_qkv, ws_h, ws_normed, ws_hid, ws_proj, ws_tscam_a, ws_tscam_y;
    int last_launches = 0;
    bool use_fused_ffn = true;   // ARD_FUSED_FFN=0 disables the fused 96-channel FFN kernel (A/B measurements)
    bool use_ln_qkv = true;      // ARD_LN_QKV=0: LayerNorm kernel + qkv GEMM instead of ln_qkv_96 (A/B measurements)
    bool use_attn_block = true;  // ARD_ATTN_BLOCK=0: ln_qkv + window_attention + proj GEMM instead of attn_block_96 (A/B measurements)
    int use_dual_gemm = 1;       // ARD_DUAL_GEMM: backward with gemm_dual (1, default) or the separate GEMMs + lambda_grad kernel (0; A/B measurements)
    int use_fused_ffn_wide = 1;    // ARD_FUSED_FFN_WIDE: 0 never, 1 C = 192 (default), 2 also C = 384, 3 also the HTSAT-base widths 128 / 256 (opt-in, see ard_api.cu)
    // training state
    DevBuf tape, p0_wT, p2_wT;
    DevBuf bw_g, bw_gs, bw_t, bw_dh, bw_gb, bw_coef, bw_gcoef, bw_gsc, bw_small;
    DevBuf bw_g3;            // fp32-grade backward: split form [hi | hi | lo] of the gradient entering a dgrad GEMM
    DevBuf tscam_wT;         // tail backward: tscam_conv weight transposed, K = 527 zero-padded to 528 [6C, 528] bf16 (built lazily)
    DevBuf bw_tail_dy, bw_tail_da;   // tail backward: dL/dy [B*32, 528] (bf16, or split [B*32, 3*528]) and dL/d im2col [B*32, 6C] fp32
    Fp32Weights fp32;        // fp32-grade split weights and workspace (ensure_fp32_weights)
    int tape_B = 0;          // batch of the forward whose activations the tape holds (0: none)
    int tape_prec = 0;       // ard_forward_args.precision of that forward: the layout of the tape and the backward schedule
    long long tape_gen = 0;  // serial number of that forward (ard_tape_generation): a backward built on an older one is refused
    int tape_tail = 0;       // tail outputs that forward computed (TAPE_* bits): a gradient for one it did not compute is refused
    // CUDA-graph replay of the inference forward (ard_api.cu): the ~110 launches of a forward cost ~1.1 ms of fixed launch /
    // ramp latency whatever the batch; replaying a captured graph removes the host side of that and most of the device side.
    struct GraphEntry {
        cudaGraphExec_t exec = nullptr;   // null: this (input, batch) was seen once and ran eagerly; captured on its next use
        unsigned long long epoch = 0, aepoch = 0;
        int launches = 0;
        unsigned long long last_use = 0;
    };
    struct GraphKey {
        const void* src;
        int B, quantize, want_ae;
        bool operator<(const GraphKey& o) const {
            if (src != o.src) return src < o.src;
            if (B != o.B) return B < o.B;
            if (quantize != o.quantize) return quantize < o.quantize;
            return want_ae < o.want_ae;
        }
    };
    std::map<GraphKey, GraphEntry> graphs;
    unsigned long long graph_epoch = 0;   // bumped when weights / injected ResiDual modules change
    unsigned long long graph_clock = 0;
    int use_graphs = 1;                   // ARD_GRAPHS=0: always launch kernel by kernel
    DevBuf g_emb, g_ae;                   // outputs of the captured forward, copied to the caller's tensors after each replay
    cudaStream_t cap_stream = nullptr;    // capture happens on a private stream (the caller's may be the legacy default stream)
    ~ard_handle() {
        for (auto& kv : graphs)
            if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
        if (cap_stream) cudaStreamDestroy(cap_stream);
    }
};


namespace ard {
enum { TAPE_FRAMEWISE = 1, TAPE_CLIPWISE = 2, TAPE_FINE = 4 };
constexpr int TSCAM_KP = 528;   // the 527 classes padded to the GEMM's K granularity
inline int C_of(const ard_handle* h, int l) { return h->cfg.embed_dim << l; }
inline int R_of(int l) { return 64 >> l; }   // tokens per side
int upload(DevBuf& b, const void* src, size_t bytes);
int upload_f32(DevBuf& b, const std::vector<float>& v);
int upload_f16(DevBuf& b, const std::vector<float>& v);
int upload_bf16(DevBuf& b, const std::vector<float>& v);
int get(const ard_handle* h, const std::string& key, size_t numel, const std::vector<float>** out);
int ensure_workspace(ard_handle* h, int B);
int ensure_fold(ard_handle* h, int l, int b, cudaStream_t s);
// training (ard_train.cu)
int ensure_tape(ard_handle* h, int B, int precision);
int encoder_backward(ard_handle* h, const ard_backward_args* a, const ard_output_grads* o, cudaStream_t s);
int tail_backward(ard_handle* h, const float* y, int ldy, const float* g_frame, const float* g_clip, const float* g_fine, const float* g_emb, int B,
                  bool fp32, float* out, cudaStream_t s);
// window-resident attention block (attn_block.cu)
int attn_block_pack(AttnBlockW& w, const std::vector<float>& qkv_w, const std::vector<float>& qkv_b, const std::vector<float>& rpb, int C, int nH);
int attn_block_pad_proj(const __nv_bfloat16* w, const float* bp, const float* bv, __nv_bfloat16* out, float* bp_eff, int C, int nH, cudaStream_t s);
int attn_block_96(const float* x, float* out, const AttnBlockW& w, const __nv_bfloat16* wp_pad, const float* bp, const float* gamma,
                  const float* beta, int B, int R, int shift, int num_sms, cudaStream_t stream);
// fp32-grade mode (fp32_mode.cu)
int ensure_fp32_weights(ard_handle* h, cudaStream_t s);   // h->fp32: forward split weights current
int split3_act(const float* in, long long ld_in, __nv_bfloat16* out, long long rows, int C, cudaStream_t s, RowAddend ext = RowAddend());
int split3_weight_host(const std::vector<float>& w, DevBuf& scratch, DevBuf& out, long long N, int K, cudaStream_t s, float scale = 1.0f,
                       long long scaled_rows = 0);
int gemm3(const __nv_bfloat16* A3, int K, const DevBuf& W3, float* out, int ldo, long long M, int N, const float* bias, int act,
          const float* r1, const float* r2, float* aux, int aux_T, long long aux_bstride, int num_sms, cudaStream_t s);
int gelu_bwd_split3(const float* g, const float* hpre, __nv_bfloat16* out3, long long rows, int N, cudaStream_t s);
int window_attention_f32_bwd(const float* qkv, const float* dout, float* dqkv, const float* bias_table, int B, int R, int C, int nH, int shift,
                             cudaStream_t s, const float* pgrad = nullptr, float pscale = 1.0f);   // pgrad: ProbGrad (ard_internal.h)
int encoder_stages_fp32(ard_handle* h, const ard_forward_args* a, float* X, float* Y, float** x_final, cudaStream_t s);
int tscam_gemm_fp32(ard_handle* h, const float* normed, float* y, int ldy, int B, cudaStream_t s);
}  // namespace ard
