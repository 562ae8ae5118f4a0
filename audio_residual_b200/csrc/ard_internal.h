// Internal host-side declarations shared by the .cu translation units of libard_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "../../include/ard.h"

namespace ard {

typedef CUresult (*PFN_cuTensorMapEncodeTiled_local)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// records the message for ard_last_error() and returns `code`
int set_error(int code, const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
#define ARD_CUDA(call)                                           \
    do {                                                         \
        if (int _rc = ::ard::check_cuda((call), #call)) return _rc; \
    } while (0)
#define ARD_TRY(call)                   \
    do {                                \
        if (int _rc = (call)) return _rc; \
    } while (0)

// ---------------------------------------------------------------- tcgen05 GEMM (gemm_tc.cu)
struct GemmArgs {
    const __nv_bfloat16* A = nullptr;  // [M, lda] row-major activations
    long long lda = 0;
    const __nv_bfloat16* W = nullptr;  // [N, ldw] row-major weights (nn.Linear layout)
    long long ldw = 0;
    void* out = nullptr;               // bf16 or fp32 [M, ldo]
    long long ldo = 0;
    int out_bf16 = 0;
    int M = 0, N = 0, K = 0;
    const float* bias = nullptr;
    int act = 0;                       // ARD_ACT_*
    const float* resid1 = nullptr;
    long long ldr1 = 0;
    const float* resid2 = nullptr;
    long long ldr2 = 0;
    float* aux = nullptr;              // fp32 copy of acc+bias before the residual adds (ResiDual/attention residual capture)
    long long ld_aux = 0;
    int aux_T = 0;
    long long aux_bstride = 0;
    int force_bn = 0;
    int force_pair = 0;                // >0: CTA-pair (cta_group::2) kernel, <0: single-CTA kernel, 0: heuristic / ARD_GEMM_PAIR
    int ab_f16 = 0;                    // A and W are fp16 instead of bf16 (the fc2 GEMM: hidden activations are fp16)
    int out_f16 = 0;                   // with out_bf16=1 and act=GELU: GELU in packed fp16, fp16 output
    const __nv_bfloat16* mul_gelu_bwd = nullptr;   // bf16 [M, ld_mul]: out = acc * gelu'(this), bf16 output only (FFN backward)
    long long ld_mul = 0;
    int splitk = 0;                    // > 1: split the K range over `splitk` partial outputs, partial s at rows [s * split_rows, +M) of `out`
    int split_rows = 0;                //      (fp32 [splitk * split_rows, ldo], split_rows % 256 == 0, >= M; plain epilogue only)
                                       //      number of partials actually written: gemm_splitk_used(K, splitk)
};
int gemm_bf16(const GemmArgs& a, int num_sms, cudaStream_t stream);
inline int gemm_splitk_used(int K, int splitk) {   // empty trailing splits are dropped
    const int num_kb = (K + 63) / 64, per = (num_kb + splitk - 1) / splitk;
    return (num_kb + per - 1) / per;
}
// Two GEMMs of one shape meeting in the epilogue (gemm_dual.cu): acc1 = A1 W1^T, acc2 = A2 W2^T, bf16 [M, ldo] output.
struct DualArgs {
    const __nv_bfloat16 *A1 = nullptr, *W1 = nullptr, *A2 = nullptr, *W2 = nullptr;   // A [M, lda] and W [N, ldw] row-major (K-major)
    long long lda1 = 0, ldw1 = 0, lda2 = 0, ldw2 = 0;
    __nv_bfloat16* out = nullptr;
    long long ldo = 0;
    int M = 0, N = 0, K = 0;
    const float* vec1 = nullptr;   // gelu_bwd: bias of GEMM 2 (fc1 bias) [N];  lambda: bias of GEMM 1 (c0) [N]
    const float* vec2 = nullptr;   // lambda: lambda [N] (zero beyond Kvalid)
    float* dlam = nullptr;         // lambda: [Kvalid], += column sums of (acc1 + vec1) * acc2
    int Kvalid = 0;
};
int gemm_dual_gelu_bwd(const DualArgs& a, int num_sms, cudaStream_t stream);   // out = acc1 * gelu'(acc2 + vec1)
int gemm_dual_lambda(const DualArgs& a, int num_sms, cudaStream_t stream);     // dlam += colsum((acc1 + vec1) * acc2), out = acc2 * vec2
int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                 uint32_t box_inner, uint32_t box_outer, int swizzle_bytes);

// ---------------------------------------------------------------- fused FFN, 96-channel stage (ffn_fused.cu)
// out = x + fc2(gelu(fc1(LayerNorm(x)))) (+ resid2); out may alias x. fc1 weights bf16, fc2 weights fp16 (hidden is fp16).
int ffn_fused_96(const float* x, const float* resid2, float* out, long long M, const float* gamma, const float* beta,
                 const __nv_bfloat16* w1, const float* b1, const __half* w2_f16, const float* b2, int num_sms, cudaStream_t stream);

// same for the 192- / 384-channel stages, weights streamed from L2 through a TMA ring (ffn_wide.cu). b1_half = 0.5 * fc1 bias.
int ffn_fused_wide(const float* x, const float* resid2, float* out, long long M, int C, const float* gamma, const float* beta,
                   const __nv_bfloat16* w1, const float* b1_half, const __half* w2_f16, const float* b2, int num_sms, cudaStream_t stream);

// ---------------------------------------------------------------- fused norm1 + qkv projection, 96-channel stage (ln_qkv.cu)
// qkv[M, 288] bf16 = LayerNorm(x[M, 96]; gamma, beta) w^T + bias
int ln_qkv_96(const float* x, const float* gamma, const float* beta, const __nv_bfloat16* w, const float* bias, __nv_bfloat16* qkv, long long M,
              int num_sms, cudaStream_t stream);

// ---------------------------------------------------------------- row-wise kernels (rowwise.cu)
// LayerNorm over the last dim C of x[rows, C] (fp32) -> bf16; two-pass variance like at::native layer_norm.
int layernorm_bf16(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, long long rows, int C, cudaStream_t s);
// PatchMerging gather (htsat.py:516-521) + LayerNorm(4C) -> bf16 [B*(H/2)*(W/2), 4C]
int merge_layernorm_bf16(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, int B, int H, int W, int C,
                         cudaStream_t s);
// fp32-grade mode: LayerNorm output written as split-bf16 rows [hi | hi | lo], 3C wide (rowwise.cu)
int layernorm_split3(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out3, long long rows, int C, cudaStream_t s);
int merge_layernorm_split3(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out3, int B, int H, int W, int C, cudaStream_t s);
// final LayerNorm + token mean (htsat.py:797, :810-811): x[B, T, C] -> emb[B, C]; optionally the normalised tokens (fp32) too
int final_norm_mean(const float* x, const float* gamma, const float* beta, float* emb, float* normed, int B, int T, int C, cudaStream_t s);
int f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, float scale, cudaStream_t s);
int fill_f32(float* p, long long n, float v, cudaStream_t s);
// backward kernels (training path)
// An fp32 addend to rows [B*T, C] stored per clip `bstride` floats apart (one block's rows b*T.. of a layers_residuals gradient
// [B, depth*T, C]: p = grad + b*T*C, bstride = depth*T*C). p == nullptr: none.
struct RowAddend {
    const float* p = nullptr;
    int T = 1;
    long long bstride = 0;
};
// out = add_scale*add + dLN(x)^T g (fp32); optional out_bf = bf16(add + dLN(x)^T g (+ ext))
int layernorm_bwd(const float* x, const float* g, const float* gamma, const float* add, float* out, long long rows, int C, cudaStream_t s,
                  float add_scale = 1.0f, __nv_bfloat16* out_bf = nullptr, RowAddend ext = RowAddend());

// ---------------------------------------------------------------- window attention (attn_window.cu)
struct AttnArgs {
    const __nv_bfloat16* qkv = nullptr;  // [B*T, 3C] token order (q already scaled by hd^-0.5)
    __nv_bfloat16* out = nullptr;        // [B*T, C] token order
    const float* bias_table = nullptr;   // [225, nH] relative_position_bias_table
    float* attn_mean = nullptr;          // optional [B*nW, nH, 64, 64] fp32; accumulates p * attn_scale
    float attn_scale = 1.0f;
    int attn_accumulate = 0;             // 0: overwrite, 1: +=
    int B = 0, H = 0, W = 0, C = 0, nH = 0, shift = 0;
};
int window_attention(const AttnArgs& a, cudaStream_t s);
// A gradient w.r.t. the attention probabilities (a loss on layers_attention, the block mean of BasicLayer.forward
// htsat.py:589-595): dP += scale * p[window, head, query, key] ([B*nW, nH, 64, 64] fp32, window order of the block). Empty when
// the kernel is instantiated without it, so those instantiations compile to the kernels without the injection.
template <bool ON> struct ProbGrad {
    const float* p;
    float scale;
};
template <> struct ProbGrad<false> {};
// pgrad (or nullptr): the probability gradient above, weighted by pscale
int window_attention_bwd(const AttnArgs& a, const __nv_bfloat16* dout, __nv_bfloat16* dqkv, cudaStream_t s, const float* pgrad = nullptr,
                         float pscale = 1.0f);

// ---------------------------------------------------------------- front end (frontend.cu)
struct MelBands {            // banded view of logmel_extractor.melW [513,64]
    const float* w = nullptr;   // [64, band_max] weights, zero padded
    const int* start = nullptr; // [64]
    const int* len = nullptr;   // [64]
    int band_max = 0;
};
int stft_logmel(const float* wave, int B, int n_samples, const float* window, const float2* twiddle, const MelBands& mel,
                const float* bn_scale, const float* bn_shift, float* out /*[B,(replicate,)frames,64]*/, long long out_clip_stride, int replicate,
                int quantize, cudaStream_t s);
int patch_embed_ln(const float* logmel /*[B,frames,64]*/, long long clip_stride, int frames, const float* bn_scale, const float* bn_shift,
                   const float* w /*[C,16]*/, const float* bias, const float* gamma, const float* beta, float* out /*[B,4096,C]*/, int B,
                   int C, cudaStream_t s);
int quantize_waveform(const float* in, float* out, long long n, cudaStream_t s);

// ---------------------------------------------------------------- heads (heads.cu)
int linear_small(const float* x, int ldx, const float* W, const float* bias, float* y, int ldy, int B, int N, int K, int act, cudaStream_t s);
int l2_normalize(const float* x, float* y, int B, int N, cudaStream_t s);
int residual_fold(const float* proj_w, const float* dmean, const float* basis, const float* lam, int C, int K, float* Mtmp,
                  __nv_bfloat16* w_out, float* b_out, cudaStream_t s, float* w_out_f32 = nullptr);
int residual_fold_batch(const float* const* proj_w, const float* const* dmean, const float* basis, const float* lam, int C, int K, float* Mtmp,
                        __nv_bfloat16* const* w_out, float* const* b_out, float* const* w_out_f32, int nb, cudaStream_t s);   // nb <= 8 blocks sharing M
int residual_matrix(const float* basis, const float* lam, int C, int K, float* M, cudaStream_t s);   // M = B^T diag(lam) B [C,C]
int tscam_im2col(const float* normed, __nv_bfloat16* A, int B, int C, cudaStream_t s);
int tscam_finish(const float* y, int ldy, float* framewise, float* clipwise, int B, int NC, cudaStream_t s);
int fine_grained(const float* normed, float* fine, int B, int C, cudaStream_t s);
// tail backward (training path): dY of the tscam conv from the pre-sigmoid y, and the token gradient in front of the final norm
int tscam_bwd_dy(const float* y, int ldy, const float* g_frame, const float* g_clip, __nv_bfloat16* dY, int Kp, int B, bool split3,
                 cudaStream_t s);
int tail_token_grad(const float* g_emb, const float* dA, const float* g_fine, float* out, int B, int C, cudaStream_t s);
// dlam[k] += sum_t coef[t,k] gcoef[t,k] (k < K; dlam may be NULL), gsc[t,k] = bf16(gcoef[t,k] lam[k]) (k < Kp); rows are Kp wide.
// split3: gsc rows are 3 Kp wide, [hi | hi | lo] of gcoef * lam (fp32-grade backward)
int lambda_grad(const float* coef, const float* gcoef, const float* lam, float* dlam, __nv_bfloat16* gsc, long long M, int K, int Kp,
                cudaStream_t s, bool split3 = false);
int head_output_tap(const __nv_bfloat16* ao, float* tap, int B, int R, int C, int nH, int shift, cudaStream_t s);   // extras.cu
int stats_accumulate(const float* x, long long rows, long long ldx, int D, double* sum, double* sumsq, cudaStream_t s);   // stats.cu

// Launch with programmatic dependent launch allowed (see pdl_wait in ard_common.cuh). ONLY for kernels that call pdl_wait()
// before their first global-memory access. ARD_PDL=0 launches them fully serialised (A/B measurements).
bool pdl_enabled();
template <class... KArgs, class... Args>
inline cudaError_t enqueue_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// launch accounting (ard_last_launch_count)
void count_launch(int n = 1);

// Per-kernel-class device timing (ard_profile_*): when enabled, every host launcher brackets its kernel with CUDA events on
// the launching stream and records the algorithmic flops / bytes of that launch. Off by default (zero overhead).
enum ProfClass { PROF_GEMM = 0, PROF_ATTN = 1, PROF_LN = 2, PROF_FRONTEND = 3, PROF_HEAD = 4, PROF_OTHER = 5, PROF_FFN = 6, PROF_NCLASS = 7 };
struct ProfScope {
    ProfScope(int cls, cudaStream_t s, double flops, double bytes);
    ~ProfScope();
    int idx;
    cudaStream_t stream;
};

}  // namespace ard
