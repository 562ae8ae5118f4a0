// fp32-grade inference mode (ard_forward_args.precision = 1): the reference computes in fp32 (hook.py:40 precision='fp32');
// north_star's second tolerance tier is rel. err <= 1e-4 against it. The bf16 tensor-core path cannot meet that (8-bit
// operand mantissas), so this mode keeps every contraction on the SAME tcgen05 GEMM kernel but feeds it 16-bit-pair operands:
//
//   x = hi + lo,  hi = bf16(x), lo = bf16(x - hi)            (16 significant bits)
//   activations [M, K] -> [hi | hi | lo]  (3K wide),  weights [N, K] -> [W_hi | W_lo | W_hi]  (3K wide)
//   one GEMM of depth 3K accumulates  hi*W_hi + hi*W_lo + lo*W_hi  in fp32 (TMEM); the dropped lo*W_lo term is 2^-18 relative.
//
// Everything between the GEMMs is fp32: LayerNorm, exact-erf GELU in the GEMM epilogue, the window attention core (SIMT fp32:
// it is 4 % of the flops), residual adds, the ResiDual fold (fp32 SIMT, then split). 3x the tensor work and ~2.5x the
// traffic of the bf16 path: a verification / high-fidelity mode, not the throughput mode.
// Training: with save_for_backward the same forward writes its intermediates to an fp32 tape (ard_train.cu), and the
// backward runs its dgrads the same way; the pieces only it needs (fp32 attention backward, gelu' into split form) are here.
#include "ard_common.cuh"
#include "ard_handle.h"

namespace ard {

// ------------------------------------------------------------------------------------------------ splitting
// in [rows, C] fp32 (row stride ld_in) -> out [rows, 3C] bf16 = [hi | hi | lo]   (activation form)
// EXT: the split of in + ext (RowAddend: a layers_residuals gradient entering the dgrad operand only)
template <bool EXT = false>
__global__ void __launch_bounds__(256) split3_act_kernel(const float* __restrict__ in, long long ld_in, __nv_bfloat16* __restrict__ out,
                                                        long long rows, int C, RowAddend ext = RowAddend()) {
    const long long total = rows * (C / 4);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / (C / 4);
        const int c = (int)(i - r * (C / 4)) * 4;
        float4 v = *reinterpret_cast<const float4*>(in + r * ld_in + c);
        if constexpr (EXT) {
            const float4 e = *reinterpret_cast<const float4*>(ext.p + (r / ext.T) * ext.bstride + (r % ext.T) * C + c);
            v.x += e.x; v.y += e.y; v.z += e.z; v.w += e.w;
        }
        const float x[4] = {v.x, v.y, v.z, v.w};
        float l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) l[k] = x[k] - __bfloat162float(__float2bfloat16_rn(x[k]));
        uint2 h, lo;
        h.x = pack_bf16x2(x[0], x[1]); h.y = pack_bf16x2(x[2], x[3]);
        lo.x = pack_bf16x2(l[0], l[1]); lo.y = pack_bf16x2(l[2], l[3]);
        __nv_bfloat16* o = out + r * (3LL * C);
        *reinterpret_cast<uint2*>(o + c) = h;
        *reinterpret_cast<uint2*>(o + C + c) = h;
        *reinterpret_cast<uint2*>(o + 2 * C + c) = lo;
    }
}
// w [N, K] fp32 -> out [N, 3K] bf16 = [hi | lo | hi]   (weight form)
__global__ void __launch_bounds__(256) split3_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, long long N, int K) {
    const long long total = N * K;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long n = i / K;
        const int k = (int)(i - n * K);
        const float x = w[i];
        const __nv_bfloat16 hi = __float2bfloat16_rn(x);
        const __nv_bfloat16 lo = __float2bfloat16_rn(x - __bfloat162float(hi));
        __nv_bfloat16* o = out + n * (3LL * K);
        o[k] = hi;
        o[K + k] = lo;
        o[2 * K + k] = hi;
    }
}

int split3_act(const float* in, long long ld_in, __nv_bfloat16* out, long long rows, int C, cudaStream_t s, RowAddend ext) {
    if (rows <= 0) return 0;
    if (C % 4 || ld_in % 4) return set_error(ARD_ERR_SHAPE, "split3: width must be a multiple of 4");
    long long blocks = (rows * (C / 4) + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ProfScope ps(PROF_OTHER, s, 0.0, (ext.p ? 14.0 : 10.0) * rows * C);
    if (ext.p) split3_act_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(in, ld_in, out, rows, C, ext);
    else split3_act_kernel<<<(unsigned)blocks, 256, 0, s>>>(in, ld_in, out, rows, C);
    return check_cuda(cudaGetLastError(), "split3_act launch");
}
static int split3_weight_dev(const float* w_dev, DevBuf& out, long long N, int K, cudaStream_t s) {
    ARD_TRY(out.ensure((size_t)N * K * 3 * 2));
    long long blocks = (N * K + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    split3_weight_kernel<<<(unsigned)blocks, 256, 0, s>>>(w_dev, out.as<__nv_bfloat16>(), N, K);
    return check_cuda(cudaGetLastError(), "split3_weight launch");
}
// host fp32 weight (optionally the first `scaled_rows` rows times `scale`: the q rows of qkv carry head_dim^-0.5) -> split device form
int split3_weight_host(const std::vector<float>& w, DevBuf& scratch, DevBuf& out, long long N, int K, cudaStream_t s, float scale,
                       long long scaled_rows) {
    const float* src = w.data();
    std::vector<float> tmp;
    if (scaled_rows > 0) {
        tmp = w;
        for (long long i = 0; i < scaled_rows * K; ++i) tmp[i] *= scale;
        src = tmp.data();
    }
    ARD_TRY(scratch.ensure((size_t)N * K * 4));
    ARD_CUDA(cudaMemcpyAsync(scratch.p, src, (size_t)N * K * 4, cudaMemcpyHostToDevice, s));
    ARD_CUDA(cudaStreamSynchronize(s));   // `tmp` / the pageable source must outlive the copy; one-time set-up cost
    return split3_weight_dev(scratch.as<float>(), out, N, K, s);
}

// ------------------------------------------------------------------------------------------------ fp32 window attention
// WindowAttention core (htsat.py:326-352) + roll / partition / reverse addressing (htsat.py:452-474) in fp32 on CUDA cores.
// One CTA of 64 threads per (clip, window, head); thread i owns query row i: q, the 64 logits / probabilities and the output
// row live in registers, K and V of the head in shared memory. qkv fp32 [B*T, 3C] token order (q pre-scaled), out fp32 [B*T, C].
template <int HD>
__global__ void __launch_bounds__(64) window_attention_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                                  const float* __restrict__ bias_table, float* __restrict__ attn,
                                                                  float attn_scale, int accumulate, float* __restrict__ tap, int R, int C,
                                                                  int nH, int shift) {
    __shared__ float Ks[64][HD + 1];
    __shared__ float Vs[64][HD + 1];
    __shared__ float bt[225];
    const int nWr = R / 8, nW = nWr * nWr;
    const int h = blockIdx.x % nH;
    const int win = (blockIdx.x / nH) % nW;
    const long long b = blockIdx.x / ((long long)nH * nW);
    const int wy = win / nWr, wx = win % nWr;
    const int i = threadIdx.x;
    const int ty = i >> 3, tx = i & 7;
    const int yr = wy * 8 + ty, xr = wx * 8 + tx;                  // coordinates in the rolled image
    int y = yr + shift, x = xr + shift;                             // source coordinates (roll by -shift, htsat.py:453)
    if (y >= R) y -= R;
    if (x >= R) x -= R;
    const long long tok = (b * R + y) * R + x;
    const float* row = qkv + tok * 3LL * C + h * HD;
    float q[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) {
        q[d] = row[d];
        Ks[i][d] = row[C + d];
        Vs[i][d] = row[2 * C + d];
    }
    for (int t = i; t < 225; t += 64) bt[t] = bias_table[t * nH + h];
    __syncthreads();
    // shift-mask region label of this token (htsat.py:414-433): slices (0,-8), (-8,-4), (-4,None) along each axis of the rolled image
    const int ly = shift == 0 ? 0 : (yr < R - 8 ? 0 : (yr < R - shift ? 1 : 2));
    const int lx = shift == 0 ? 0 : (xr < R - 8 ? 0 : (xr < R - shift ? 1 : 2));
    const int label = ly * 3 + lx;
    float sc[64];
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 64; ++j) {
        float a = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) a = fmaf(q[d], Ks[j][d], a);
        const int jy = j >> 3, jx = j & 7;
        a += bt[(ty - jy + 7) * 15 + (tx - jx + 7)];               // relative_position_index, htsat.py:301-316
        if (shift != 0) {
            const int yj = wy * 8 + jy, xj = wx * 8 + jx;
            const int lj = (yj < R - 8 ? 0 : (yj < R - shift ? 1 : 2)) * 3 + (xj < R - 8 ? 0 : (xj < R - shift ? 1 : 2));
            if (lj != label) a += -100.0f;                          // htsat.py:432-433
        }
        sc[j] = a;
        m = fmaxf(m, a);
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 64; ++j) {
        sc[j] = expf(sc[j] - m);
        sum += sc[j];
    }
    const float inv = 1.0f / sum;
    float o[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) o[d] = 0.f;
#pragma unroll
    for (int j = 0; j < 64; ++j) {
        sc[j] *= inv;
#pragma unroll
        for (int d = 0; d < HD; ++d) o[d] = fmaf(sc[j], Vs[j][d], o[d]);
    }
    float* op = out + tok * (long long)C + h * HD;
#pragma unroll
    for (int d = 0; d < HD; ++d) op[d] = o[d];
    const long long wh = ((b * nW + win) * nH + h) * 64 + i;        // (window, head, query row)
    if (attn != nullptr) {
        float* ap = attn + wh * 64;
#pragma unroll
        for (int j = 0; j < 64; ++j) ap[j] = accumulate ? ap[j] + sc[j] * attn_scale : sc[j] * attn_scale;
    }
    if (tap != nullptr) {
        float* tp = tap + wh * HD;
#pragma unroll
        for (int d = 0; d < HD; ++d) tp[d] = o[d];
    }
}

static int window_attention_f32(const float* qkv, float* out, const float* bias_table, float* attn, float attn_scale, int accumulate, float* tap,
                                int B, int R, int C, int nH, int shift, cudaStream_t s) {
    const int hd = C / nH;
    const int nW = (R / 8) * (R / 8);
    const long long ctas = (long long)B * nW * nH;
    if (ctas > 0x7fffffffLL) return set_error(ARD_ERR_SHAPE, "window_attention_f32: batch too large");
    const int sh = R > 8 ? shift : 0;                               // htsat.py:393-396
    ProfScope ps(PROF_ATTN, s, 4.0 * 64 * 64 * hd * ctas, 16.0 * B * R * R * C);
    if (hd == 24) window_attention_f32_kernel<24><<<(unsigned)ctas, 64, 0, s>>>(qkv, out, bias_table, attn, attn_scale, accumulate, tap, R, C, nH, sh);
    else if (hd == 32) window_attention_f32_kernel<32><<<(unsigned)ctas, 64, 0, s>>>(qkv, out, bias_table, attn, attn_scale, accumulate, tap, R, C, nH, sh);
    else return set_error(ARD_ERR_SHAPE, "window_attention_f32: head dim %d unsupported (24 or 32)", hd);
    return check_cuda(cudaGetLastError(), "window_attention_f32 launch");
}

// ------------------------------------------------------------------------------------------------ fp32 window attention backward
// Autograd of the kernel above w.r.t. qkv (loss.backward() through htsat.py:326-352), fp32 on CUDA cores with the same CTA
// decomposition and addressing. Thread i recomputes probability row i, then
//   dP = dO V^T,  delta = rowsum(dP . P),  dS = P . (dP - delta),  dQ = dS K          (row i: registers)
//   dK = dS^T Q,  dV = P^T dO                                                          (key row i: columns of P / dS via smem)
// qkv fp32 [B*T, 3C] token order (q pre-scaled), dout fp32 [B*T, C] -> dqkv fp32 [B*T, 3C] token order (d of the pre-scaled q).
template <int HD>
constexpr int attn_f32_bwd_smem() { return (4 * 64 * (HD + 1) + 2 * 64 * 65 + 225) * 4; }

// GP: a probability gradient (ProbGrad) is added to dP before delta.
template <int HD, bool GP = false>
__global__ void __launch_bounds__(64) window_attention_f32_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ dout,
                                                                      float* __restrict__ dqkv, const float* __restrict__ bias_table, int R,
                                                                      int C, int nH, int shift, ProbGrad<GP> pg = {}) {
    extern __shared__ float sm[];
    float (*Qs)[HD + 1] = reinterpret_cast<float (*)[HD + 1]>(sm);
    float (*Ks)[HD + 1] = Qs + 64;
    float (*Vs)[HD + 1] = Ks + 64;
    float (*Os)[HD + 1] = Vs + 64;                                  // dO
    float (*Ps)[65] = reinterpret_cast<float (*)[65]>(sm + 4 * 64 * (HD + 1));
    float (*Ds)[65] = Ps + 64;                                      // dS
    float* bt = sm + 4 * 64 * (HD + 1) + 2 * 64 * 65;
    const int nWr = R / 8, nW = nWr * nWr;
    const int h = blockIdx.x % nH;
    const int win = (blockIdx.x / nH) % nW;
    const long long b = blockIdx.x / ((long long)nH * nW);
    const int wy = win / nWr, wx = win % nWr;
    const int i = threadIdx.x;
    const int ty = i >> 3, tx = i & 7;
    const int yr = wy * 8 + ty, xr = wx * 8 + tx;
    int y = yr + shift, x = xr + shift;
    if (y >= R) y -= R;
    if (x >= R) x -= R;
    const long long tok = (b * R + y) * R + x;
    const float* row = qkv + tok * 3LL * C + h * HD;
    const float* grow = dout + tok * (long long)C + h * HD;
    float q[HD], go[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) {
        q[d] = row[d];
        Qs[i][d] = q[d];
        Ks[i][d] = row[C + d];
        Vs[i][d] = row[2 * C + d];
        go[d] = grow[d];
        Os[i][d] = go[d];
    }
    for (int t = i; t < 225; t += 64) bt[t] = bias_table[t * nH + h];
    __syncthreads();
    const int ly = shift == 0 ? 0 : (yr < R - 8 ? 0 : (yr < R - shift ? 1 : 2));
    const int lx = shift == 0 ? 0 : (xr < R - 8 ? 0 : (xr < R - shift ? 1 : 2));
    const int label = ly * 3 + lx;
    float sc[64];
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 64; ++j) {                                  // logits exactly as the forward kernel forms them
        float a = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) a = fmaf(q[d], Ks[j][d], a);
        const int jy = j >> 3, jx = j & 7;
        a += bt[(ty - jy + 7) * 15 + (tx - jx + 7)];
        if (shift != 0) {
            const int yj = wy * 8 + jy, xj = wx * 8 + jx;
            const int lj = (yj < R - 8 ? 0 : (yj < R - shift ? 1 : 2)) * 3 + (xj < R - 8 ? 0 : (xj < R - shift ? 1 : 2));
            if (lj != label) a += -100.0f;
        }
        sc[j] = a;
        m = fmaxf(m, a);
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 64; ++j) {
        sc[j] = expf(sc[j] - m);
        sum += sc[j];
    }
    const float inv = 1.0f / sum;
    float delta = 0.f;
    const float* gp = nullptr;
    if constexpr (GP) gp = pg.p + ((b * nW + win) * nH + h) * 4096 + i * 64;   // (window, head, query row i)
#pragma unroll
    for (int j = 0; j < 64; ++j) {                                  // P to smem, dP into sc
        const float p = sc[j] * inv;
        Ps[i][j] = p;
        float dp = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) dp = fmaf(go[d], Vs[j][d], dp);
        if constexpr (GP) dp = fmaf(pg.scale, __ldg(gp + j), dp);
        sc[j] = dp;
        delta = fmaf(dp, p, delta);
    }
    float dq[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) dq[d] = 0.f;
#pragma unroll
    for (int j = 0; j < 64; ++j) {
        const float ds = Ps[i][j] * (sc[j] - delta);
        Ds[i][j] = ds;
#pragma unroll
        for (int d = 0; d < HD; ++d) dq[d] = fmaf(ds, Ks[j][d], dq[d]);
    }
    float* op = dqkv + tok * 3LL * C + h * HD;
#pragma unroll
    for (int d = 0; d < HD; ++d) op[d] = dq[d];
    __syncthreads();
    // thread i now owns KEY row i (the same token): column sums over the 64 query rows
    float dk[HD], dv[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) { dk[d] = 0.f; dv[d] = 0.f; }
    for (int r = 0; r < 64; ++r) {
        const float ds = Ds[r][i], p = Ps[r][i];
#pragma unroll
        for (int d = 0; d < HD; ++d) {
            dk[d] = fmaf(ds, Qs[r][d], dk[d]);
            dv[d] = fmaf(p, Os[r][d], dv[d]);
        }
    }
#pragma unroll
    for (int d = 0; d < HD; ++d) {
        op[C + d] = dk[d];
        op[2 * C + d] = dv[d];
    }
}

int window_attention_f32_bwd(const float* qkv, const float* dout, float* dqkv, const float* bias_table, int B, int R, int C, int nH, int shift,
                             cudaStream_t s, const float* pgrad, float pscale) {
    if (B <= 0 || R <= 0 || R % 8 || nH <= 0 || C % nH)
        return set_error(ARD_ERR_SHAPE, "window_attention_f32_bwd: unsupported shape B=%d R=%d C=%d nH=%d", B, R, C, nH);
    const int hd = C / nH;
    const int nW = (R / 8) * (R / 8);
    const long long ctas = (long long)B * nW * nH;
    if (ctas > 0x7fffffffLL) return set_error(ARD_ERR_SHAPE, "window_attention_f32_bwd: batch too large");
    const int sh = R > 8 ? shift : 0;                               // htsat.py:393-396, as the forward launcher
    static bool attr_set = false;
    if (!attr_set) {
        ARD_CUDA(cudaFuncSetAttribute(window_attention_f32_bwd_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_f32_bwd_smem<24>()));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_f32_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_f32_bwd_smem<32>()));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_f32_bwd_kernel<24, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_f32_bwd_smem<24>()));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_f32_bwd_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_f32_bwd_smem<32>()));
        attr_set = true;
    }
    ProfScope ps(PROF_ATTN, s, 10.0 * 64 * 64 * hd * ctas, 28.0 * B * R * R * C + (pgrad ? 16384.0 * ctas : 0.0));
    if (pgrad) {
        const ProbGrad<true> pg{pgrad, pscale};
        if (hd == 24)
            window_attention_f32_bwd_kernel<24, true><<<(unsigned)ctas, 64, attn_f32_bwd_smem<24>(), s>>>(qkv, dout, dqkv, bias_table, R, C, nH, sh, pg);
        else if (hd == 32)
            window_attention_f32_bwd_kernel<32, true><<<(unsigned)ctas, 64, attn_f32_bwd_smem<32>(), s>>>(qkv, dout, dqkv, bias_table, R, C, nH, sh, pg);
        else return set_error(ARD_ERR_SHAPE, "window_attention_f32_bwd: head dim %d unsupported (24 or 32)", hd);
        return check_cuda(cudaGetLastError(), "window_attention_f32_bwd launch");
    }
    if (hd == 24)
        window_attention_f32_bwd_kernel<24><<<(unsigned)ctas, 64, attn_f32_bwd_smem<24>(), s>>>(qkv, dout, dqkv, bias_table, R, C, nH, sh);
    else if (hd == 32)
        window_attention_f32_bwd_kernel<32><<<(unsigned)ctas, 64, attn_f32_bwd_smem<32>(), s>>>(qkv, dout, dqkv, bias_table, R, C, nH, sh);
    else return set_error(ARD_ERR_SHAPE, "window_attention_f32_bwd: head dim %d unsupported (24 or 32)", hd);
    return check_cuda(cudaGetLastError(), "window_attention_f32_bwd launch");
}

// FFN backward through the exact-erf GELU (htsat.py:151): dh = g * gelu'(hpre), g and hpre fp32 [rows, N], written straight
// into the split activation form [hi | hi | lo] ([rows, 3N] bf16) that the next dgrad GEMM reads
__global__ void __launch_bounds__(256) gelu_bwd_split3_kernel(const float* __restrict__ g, const float* __restrict__ hpre,
                                                             __nv_bfloat16* __restrict__ out, long long rows, int N) {
    const long long total = rows * (N / 4);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / (N / 4);
        const int c = (int)(i - r * (N / 4)) * 4;
        const float4 gv = *reinterpret_cast<const float4*>(g + r * N + c);
        const float4 hv = *reinterpret_cast<const float4*>(hpre + r * N + c);
        const float x[4] = {gv.x * gelu_erf_grad(hv.x), gv.y * gelu_erf_grad(hv.y), gv.z * gelu_erf_grad(hv.z), gv.w * gelu_erf_grad(hv.w)};
        float l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) l[k] = x[k] - __bfloat162float(__float2bfloat16_rn(x[k]));
        uint2 hi, lo;
        hi.x = pack_bf16x2(x[0], x[1]); hi.y = pack_bf16x2(x[2], x[3]);
        lo.x = pack_bf16x2(l[0], l[1]); lo.y = pack_bf16x2(l[2], l[3]);
        __nv_bfloat16* o = out + r * (3LL * N);
        *reinterpret_cast<uint2*>(o + c) = hi;
        *reinterpret_cast<uint2*>(o + N + c) = hi;
        *reinterpret_cast<uint2*>(o + 2 * N + c) = lo;
    }
}
int gelu_bwd_split3(const float* g, const float* hpre, __nv_bfloat16* out3, long long rows, int N, cudaStream_t s) {
    if (rows <= 0) return 0;
    if (N % 4) return set_error(ARD_ERR_SHAPE, "gelu_bwd_split3: width must be a multiple of 4");
    long long blocks = (rows * (N / 4) + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ProfScope ps(PROF_OTHER, s, 30.0 * rows * N, 14.0 * rows * N);
    gelu_bwd_split3_kernel<<<(unsigned)blocks, 256, 0, s>>>(g, hpre, out3, rows, N);
    return check_cuda(cudaGetLastError(), "gelu_bwd_split3 launch");
}

// tscam_conv im2col (heads.cu::tscam_im2col_kernel) straight into the split activation form [hi | hi | lo] of width 3 * 6C
__global__ void tscam_im2col_split3_kernel(const float* __restrict__ normed, __nv_bfloat16* __restrict__ A3, int B, int C) {
    const long long K6 = 6LL * C;
    const long long total = (long long)B * 32 * K6;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int kw = (int)(i % 3);
        const int fb = (int)((i / 3) % 2);
        const int c = (int)((i / 6) % C);
        const long long row = i / K6;
        const int Tp = (int)(row % 32);
        const long long b = row / 32;
        const int tt = Tp + kw - 1;
        float v = 0.f;
        if (tt >= 0 && tt < 32) {
            const int gq = tt >> 3, t = tt & 7;
            v = normed[(b * 64 + (gq * 2 + fb) * 8 + t) * C + c];
        }
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
        const long long col = i - row * K6;
        __nv_bfloat16* o = A3 + row * 3 * K6;
        o[col] = hi;
        o[K6 + col] = hi;
        o[2 * K6 + col] = lo;
    }
}

// ------------------------------------------------------------------------------------------------ weights
int ensure_fp32_weights(ard_handle* h, cudaStream_t s) {
    Fp32Weights& w = h->fp32;
    if (w.epoch == h->graph_epoch && !w.blocks.empty()) return 0;
    w.blocks.resize(h->nlayers);
    w.merge3.resize(h->nlayers);
    w.mergeT3.resize(h->nlayers);
    const std::vector<float>* v = nullptr;
    for (int l = 0; l < h->nlayers; ++l) {
        const int C = C_of(h, l), nH = h->cfg.num_heads[l];
        w.blocks[l].resize(h->cfg.depths[l]);
        for (int b = 0; b < h->cfg.depths[l]; ++b) {
            char pfx[64];
            snprintf(pfx, sizeof(pfx), "layers.%d.blocks.%d.", l, b);
            const std::string p(pfx);
            Fp32BlockW& fw = w.blocks[l][b];
            ARD_TRY(get(h, p + "attn.qkv.weight", (size_t)3 * C * C, &v));
            ARD_TRY(split3_weight_host(*v, w.scratch, fw.qkv3, 3LL * C, C, s, 1.0f / sqrtf((float)(C / nH)), C));   // q rows pre-scaled (htsat.py:295,331)
            ARD_TRY(get(h, p + "attn.proj.weight", (size_t)C * C, &v));
            ARD_TRY(split3_weight_host(*v, w.scratch, fw.proj3, C, C, s));
            ARD_TRY(get(h, p + "mlp.fc1.weight", (size_t)4 * C * C, &v));
            ARD_TRY(split3_weight_host(*v, w.scratch, fw.fc13, 4LL * C, C, s));
            ARD_TRY(get(h, p + "mlp.fc2.weight", (size_t)4 * C * C, &v));
            ARD_TRY(split3_weight_host(*v, w.scratch, fw.fc23, C, 4 * C, s));
        }
        if (l < h->nlayers - 1) {
            char key[64];
            snprintf(key, sizeof(key), "layers.%d.downsample.reduction.weight", l);
            ARD_TRY(get(h, key, (size_t)8 * C * C, &v));
            ARD_TRY(split3_weight_host(*v, w.scratch, w.merge3[l], 2LL * C, 4 * C, s));
        }
    }
    if (h->host.count("tscam_conv.weight")) {
        const int NF = C_of(h, h->nlayers - 1);
        ARD_TRY(get(h, "tscam_conv.weight", (size_t)ARD_CLASS_NUM * NF * 6, &v));
        ARD_TRY(split3_weight_host(*v, w.scratch, w.tscam3, ARD_CLASS_NUM, 6 * NF, s));
    }
    w.epoch = h->graph_epoch;
    return 0;
}

int gemm3(const __nv_bfloat16* A3, int K, const DevBuf& W3, float* out, int ldo, long long M, int N, const float* bias, int act,
          const float* r1, const float* r2, float* aux, int aux_T, long long aux_bstride, int num_sms, cudaStream_t s) {
    GemmArgs g;
    g.A = A3; g.lda = 3LL * K; g.W = W3.as<__nv_bfloat16>(); g.ldw = 3LL * K; g.out = out; g.ldo = ldo;
    g.M = (int)M; g.N = N; g.K = 3 * K; g.bias = bias; g.act = act;
    g.resid1 = r1; g.ldr1 = ldo; g.resid2 = r2; g.ldr2 = ldo;
    if (aux) { g.aux = aux; g.ld_aux = N; g.aux_T = aux_T; g.aux_bstride = aux_bstride; }
    g.force_pair = -1;
    return gemm_bf16(g, num_sms, s);
}

// Where one block of the fp32-grade forward reads and writes. Inference: s = out = X, x1 = x3 = Y (scratch), qkv / ao in the
// workspace. Training: the block's tape slots (ard_train.cu), so the backward finds every intermediate it needs.
struct Fp32BlockIO {
    float *s, *x1, *x3, *out, *qkv, *ao;
};

// One Swin block (plain htsat.py:439-482 or patched src/residual.py:58-98) in the fp32-grade mode.
static int run_block_fp32(ard_handle* h, Fp32Weights& w, int l, int b, int B, const Fp32BlockIO& io, float* attn_out, float attn_scale,
                          int attn_acc, float* res_out, long long res_bstride, float* head_tap, cudaStream_t s) {
    BlockW& bw = h->layers[l].blocks[b];
    Fp32BlockW& fw = w.blocks[l][b];
    const int C = C_of(h, l), R = R_of(l), T = R * R, nH = h->cfg.num_heads[l];
    const long long M = (long long)B * T;
    float* Hf = w.qkvf.as<float>();
    __nv_bfloat16* S3 = w.s3.as<__nv_bfloat16>();
    const int shift = (b % 2 == 0) ? 0 : 4;
    ARD_TRY(layernorm_split3(io.s, bw.ln1_g.as<float>(), bw.ln1_b.as<float>(), S3, M, C, s));
    ARD_TRY(gemm3(S3, C, fw.qkv3, io.qkv, 3 * C, M, 3 * C, bw.qkv_b.as<float>(), ARD_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));
    ARD_TRY(window_attention_f32(io.qkv, io.ao, bw.rpb.as<float>(), attn_out, attn_scale, attn_acc, head_tap, B, R, C, nH, shift, s));
    ARD_TRY(split3_act(io.ao, C, S3, M, C, s));
    const DevBuf* pw = &fw.proj3;
    const float* pb = bw.proj_b.as<float>();
    if (bw.has_res) {   // the folded projection depends on the current lambda: re-split per call (C^2 elements)
        ARD_TRY(ensure_fold(h, l, b, s));
        ARD_TRY(split3_weight_dev(bw.proj_w_fold_f32.as<float>(), w.fold3, C, C, s));
        pw = &w.fold3;
        pb = bw.proj_b_fold.as<float>();
    }
    // x1 = s + r,  aux = r = residual_x (post-ResiDual for patched blocks)
    ARD_TRY(gemm3(S3, C, *pw, io.x1, C, M, C, pb, ARD_ACT_NONE, io.s, nullptr, res_out, T, res_bstride, h->num_sms, s));
    auto ffn = [&](const float* in, float* out, const float* r2) -> int {   // out = in + mlp(norm2(in)) (+ r2)
        ARD_TRY(layernorm_split3(in, bw.ln2_g.as<float>(), bw.ln2_b.as<float>(), S3, M, C, s));
        ARD_TRY(gemm3(S3, C, fw.fc13, Hf, 4 * C, M, 4 * C, bw.fc1_b.as<float>(), ARD_ACT_GELU, nullptr, nullptr, nullptr, 0, 0, h->num_sms, s));
        ARD_TRY(split3_act(Hf, 4 * C, S3, M, 4 * C, s));
        return gemm3(S3, 4 * C, fw.fc23, out, C, M, C, bw.fc2_b.as<float>(), ARD_ACT_NONE, in, r2, nullptr, 0, 0, h->num_sms, s);
    };
    if (!bw.has_res) return ffn(io.x1, io.out, nullptr);             // htsat.py:480
    ARD_TRY(ffn(io.x1, io.x3, io.s));                                // x3 = shortcut + (x1 + mlp(norm2(x1)))   src/residual.py:93,95
    return ffn(io.x3, io.out, nullptr);                              // x4 = x3 + mlp(norm2(x3))                src/residual.py:96
}

// Swin stages of the forward in the fp32-grade mode; X holds the patch-embed output (front end is fp32 already). With
// a->save_for_backward, X is the tape's first slot and every block writes its tape slots (ensure_tape(h, B, 1) ran).
int encoder_stages_fp32(ard_handle* h, const ard_forward_args* a, float* X, float* Y, float** x_final, cudaStream_t s) {
    ARD_TRY(ensure_fp32_weights(h, s));
    Fp32Weights& w = h->fp32;
    const int B = a->B;
    const bool train = a->save_for_backward != 0;
    const size_t MC = (size_t)B * 4096 * h->cfg.embed_dim;
    ARD_TRY(w.qkvf.ensure(MC * 16));
    ARD_TRY(w.aof.ensure(MC * 4));
    ARD_TRY(w.s3.ensure(MC * 24));
    for (int l = 0; l < h->nlayers; ++l) {
        const int C = C_of(h, l), R = R_of(l), T = R * R, depth = h->cfg.depths[l];
        for (int b = 0; b < depth; ++b) {
            float* res = a->layers_residuals[l] ? a->layers_residuals[l] + (long long)b * T * C : nullptr;
            float* tap = a->head_outputs[l] ? a->head_outputs[l] + (long long)b * B * T * C : nullptr;
            const BlockW& bw = h->layers[l].blocks[b];
            const Fp32BlockIO io = train ? Fp32BlockIO{bw.t_s, bw.t_x1, bw.t_x3, bw.t_out, bw.t_qkvf, bw.t_aof}
                                         : Fp32BlockIO{X, Y, Y, X, w.qkvf.as<float>(), w.aof.as<float>()};
            ARD_TRY(run_block_fp32(h, w, l, b, B, io, a->layers_attention[l], 1.0f / depth, b > 0, res, (long long)depth * T, tap, s));
            if (train) X = bw.t_out;
        }
        if (l < h->nlayers - 1) {   // PatchMerging (htsat.py:505-526)
            float* mout = train ? h->layers[l + 1].blocks[0].t_s : Y;
            ARD_TRY(merge_layernorm_split3(X, h->layers[l].mg_g.as<float>(), h->layers[l].mg_b.as<float>(), w.s3.as<__nv_bfloat16>(), B, R, R, C, s));
            ARD_TRY(gemm3(w.s3.as<__nv_bfloat16>(), 4 * C, w.merge3[l], mout, 2 * C, (long long)B * (T / 4), 2 * C, nullptr, ARD_ACT_NONE, nullptr,
                          nullptr, nullptr, 0, 0, h->num_sms, s));
            if (train) X = mout;
            else { Y = X; X = mout; }
        }
    }
    *x_final = X;
    return 0;
}

// tscam_conv (htsat.py:813-816) as a split GEMM: y [B*32, ldy] fp32
int tscam_gemm_fp32(ard_handle* h, const float* normed, float* y, int ldy, int B, cudaStream_t s) {
    Fp32Weights& w = h->fp32;
    const int NF = C_of(h, h->nlayers - 1);
    if (!w.tscam3.p) return set_error(ARD_ERR_STATE, "tscam_conv weights were never set");
    ARD_TRY(w.s3.ensure((size_t)B * 32 * 18 * NF * 2));
    tscam_im2col_split3_kernel<<<148 * 8, 256, 0, s>>>(normed, w.s3.as<__nv_bfloat16>(), B, NF);
    ARD_TRY(check_cuda(cudaGetLastError(), "tscam_im2col_split3 launch"));
    return gemm3(w.s3.as<__nv_bfloat16>(), 6 * NF, w.tscam3, y, ldy, (long long)B * 32, ARD_CLASS_NUM, h->tscam_b.as<float>(), ARD_ACT_NONE, nullptr,
                 nullptr, nullptr, 0, 0, h->num_sms, s);
}

}  // namespace ard
