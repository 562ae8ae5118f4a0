// Row-wise HBM-bound kernels: LayerNorm (-> bf16 GEMM operand), PatchMerging gather + LayerNorm, final norm + token mean,
// dtype conversion, waveform quantisation. One warp per row, the row is held in registers, loads are coalesced/vectorised.
#include "ard_common.cuh"
#include "ard_internal.h"

namespace ard {

constexpr float LN_EPS = 1e-5f;

ARD_DEVINL float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int VEC>
ARD_DEVINL void load_vec(const float* p, float* r) {
    if constexpr (VEC == 4) {
        float4 t = *reinterpret_cast<const float4*>(p);
        r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
    } else if constexpr (VEC == 2) {
        float2 t = *reinterpret_cast<const float2*>(p);
        r[0] = t.x; r[1] = t.y;
    } else {
        r[0] = *p;
    }
}
template <int VEC>
ARD_DEVINL void store_bf16_vec(__nv_bfloat16* p, const float* r) {
    if constexpr (VEC == 4) {
        uint2 u;
        u.x = pack_bf16x2(r[0], r[1]);
        u.y = pack_bf16x2(r[2], r[3]);
        *reinterpret_cast<uint2*>(p) = u;
    } else if constexpr (VEC == 2) {
        *reinterpret_cast<uint32_t*>(p) = pack_bf16x2(r[0], r[1]);
    } else {
        *p = __float2bfloat16_rn(r[0]);
    }
}

// fp32-grade mode: a value is carried as two bf16 terms, hi = bf16(x), lo = bf16(x - hi) (16 significant bits); an activation
// row of width C is laid out [hi | hi | lo] (3C wide) so that ONE GEMM against the weight rows [W_hi | W_lo | W_hi] accumulates
// hi*hi + hi*lo + lo*hi in fp32 (the dropped lo*lo term is 2^-18 relative).
template <int VEC>
ARD_DEVINL void store_split3_vec(__nv_bfloat16* row_base, int C, int e, const float* r) {
    float lo[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) lo[k] = r[k] - __bfloat162float(__float2bfloat16_rn(r[k]));
    store_bf16_vec<VEC>(row_base + e, r);
    store_bf16_vec<VEC>(row_base + C + e, r);
    store_bf16_vec<VEC>(row_base + 2 * C + e, lo);
}

// Row r of the logical [rows, C] matrix; element offset e (multiple of VEC) -> source pointer.
struct PlainRows {
    const float* x;
    int C;
    ARD_DEVINL const float* at(long long row, int e) const { return x + row * C + e; }
};
// PatchMerging.forward htsat.py:516-521: logical row (b, i, j) of width 4*Cin = [x(2i,2j), x(2i+1,2j), x(2i,2j+1), x(2i+1,2j+1)]
struct MergeRows {
    const float* x;
    int H, W, Cin;
    ARD_DEVINL const float* at(long long row, int e) const {
        const int W2 = W >> 1, H2 = H >> 1;
        const int j = (int)(row % W2);
        const long long t = row / W2;
        const int i = (int)(t % H2);
        const long long b = t / H2;
        const int s = e / Cin, c = e - s * Cin;
        const int hh = 2 * i + (s & 1), ww = 2 * j + (s >> 1);
        return x + ((b * H + hh) * W + ww) * (long long)Cin + c;
    }
};

template <int VEC, int NV, class Rows, bool SPLIT3 = false>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(Rows rows, const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            __nv_bfloat16* __restrict__ out, long long nrows) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int C = 32 * VEC * NV;
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= nrows) return;
    float v[NV][VEC];
#pragma unroll
    for (int i = 0; i < NV; ++i) load_vec<VEC>(rows.at(row, (i * 32 + lane) * VEC), v[i]);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) s += v[i][k];
    const float mean = warp_sum(s) * (1.0f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            const float d = v[i][k] - mean;
            q = fmaf(d, d, q);
        }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / C) + LN_EPS);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int e = (i * 32 + lane) * VEC;
        float g[VEC], b[VEC], o[VEC];
        load_vec<VEC>(gamma + e, g);
        load_vec<VEC>(beta + e, b);
#pragma unroll
        for (int k = 0; k < VEC; ++k) o[k] = fmaf((v[i][k] - mean) * rstd, g[k], b[k]);
        if constexpr (SPLIT3) store_split3_vec<VEC>(out + row * (3 * C), C, e, o);
        else store_bf16_vec<VEC>(out + row * C + e, o);
    }
}

template <class Rows, bool SPLIT3 = false>
static int launch_ln(Rows rows, const float* gamma, const float* beta, __nv_bfloat16* out, long long nrows, int C, cudaStream_t s) {
    const int wpb = 8;
    const unsigned grid = (unsigned)((nrows + wpb - 1) / wpb);
    ProfScope ps(PROF_LN, s, 8.0 * nrows * C, (SPLIT3 ? 10.0 : 6.0) * nrows * C);
#define ARD_LN_CASE(c, vec, nv) \
    case c: ARD_CUDA(enqueue_pdl(layernorm_rows_kernel<vec, nv, Rows, SPLIT3>, dim3(grid), dim3(wpb * 32), 0, s, rows, gamma, beta, out, nrows)); break;
    switch (C) {
        ARD_LN_CASE(96, 1, 3)
        ARD_LN_CASE(128, 4, 1)
        ARD_LN_CASE(192, 2, 3)
        ARD_LN_CASE(256, 4, 2)
        ARD_LN_CASE(384, 4, 3)
        ARD_LN_CASE(512, 4, 4)
        ARD_LN_CASE(768, 4, 6)
        ARD_LN_CASE(1024, 4, 8)
        ARD_LN_CASE(1536, 4, 12)
        ARD_LN_CASE(2048, 4, 16)
        default: return set_error(ARD_ERR_SHAPE, "layernorm: unsupported width C=%d", C);
    }
#undef ARD_LN_CASE
    return check_cuda(cudaGetLastError(), "layernorm launch");
}

int layernorm_bf16(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, long long rows, int C, cudaStream_t s) {
    if (rows <= 0) return 0;
    return launch_ln(PlainRows{x, C}, gamma, beta, out, rows, C, s);
}

int merge_layernorm_bf16(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out, int B, int H, int W, int C,
                         cudaStream_t s) {
    if ((H & 1) || (W & 1)) return set_error(ARD_ERR_SHAPE, "x size (%d*%d) are not even.", H, W);  // htsat.py:512
    const long long rows = (long long)B * (H / 2) * (W / 2);
    return launch_ln(MergeRows{x, H, W, C}, gamma, beta, out, rows, 4 * C, s);
}

// fp32-grade mode: LayerNorm output as split-bf16 rows [hi | hi | lo] (3C wide)
int layernorm_split3(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out3, long long rows, int C, cudaStream_t s) {
    if (rows <= 0) return 0;
    return launch_ln<PlainRows, true>(PlainRows{x, C}, gamma, beta, out3, rows, C, s);
}
int merge_layernorm_split3(const float* x, const float* gamma, const float* beta, __nv_bfloat16* out3, int B, int H, int W, int C, cudaStream_t s) {
    if ((H & 1) || (W & 1)) return set_error(ARD_ERR_SHAPE, "x size (%d*%d) are not even.", H, W);  // htsat.py:512
    const long long rows = (long long)B * (H / 2) * (W / 2);
    return launch_ln<MergeRows, true>(MergeRows{x, H, W, C}, gamma, beta, out3, rows, 4 * C, s);
}

// ---------------------------------------------------------------------------------------------- final norm + token mean
// forward_features tail, htsat.py:797 (self.norm) and :810-811 (avgpool over all tokens) : x[B, T, C] -> emb[B, C].
// One CTA per clip, one warp per token (T = 64 tokens, 8 warps x 8 tokens).
template <int VEC, int NV>
__global__ void __launch_bounds__(256) final_norm_mean_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, float* __restrict__ emb,
                                                             float* __restrict__ normed, int T) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int C = 32 * VEC * NV;
    __shared__ float part[8][C];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = blockIdx.x;
    float acc[NV][VEC];
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[i][k] = 0.f;
    for (int t = warp; t < T; t += 8) {
        const float* xr = x + (b * T + t) * C;
        float v[NV][VEC];
#pragma unroll
        for (int i = 0; i < NV; ++i) load_vec<VEC>(xr + (i * 32 + lane) * VEC, v[i]);
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
            for (int k = 0; k < VEC; ++k) s += v[i][k];
        const float mean = warp_sum(s) * (1.0f / C);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                const float d = v[i][k] - mean;
                q = fmaf(d, d, q);
            }
        const float rstd = rsqrtf(warp_sum(q) * (1.0f / C) + LN_EPS);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int e = (i * 32 + lane) * VEC;
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                const float o = fmaf((v[i][k] - mean) * rstd, __ldg(gamma + e + k), __ldg(beta + e + k));
                acc[i][k] += o;
                if (normed) normed[(b * T + t) * C + e + k] = o;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) part[warp][(i * 32 + lane) * VEC + k] = acc[i][k];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += part[w][c];
        emb[b * C + c] = s / (float)T;
    }
}

int final_norm_mean(const float* x, const float* gamma, const float* beta, float* emb, float* normed, int B, int T, int C, cudaStream_t s) {
    if (B <= 0) return 0;
    ProfScope ps(PROF_HEAD, s, 8.0 * B * T * C, 4.0 * B * T * C * (normed ? 2 : 1));
    switch (C) {
        case 768: ARD_CUDA(enqueue_pdl(final_norm_mean_kernel<4, 6>, dim3(B), dim3(256), 0, s, x, gamma, beta, emb, normed, T)); break;
        case 1024: ARD_CUDA(enqueue_pdl(final_norm_mean_kernel<4, 8>, dim3(B), dim3(256), 0, s, x, gamma, beta, emb, normed, T)); break;
        default: return set_error(ARD_ERR_SHAPE, "final norm: unsupported width C=%d", C);
    }
    return check_cuda(cudaGetLastError(), "final_norm_mean launch");
}

// ---------------------------------------------------------------------------------------------- conversions
__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n, float scale) {
    long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const long long stride = (long long)gridDim.x * blockDim.x * 4;
    for (; i + 3 < n; i += stride) {
        const float4 v = *reinterpret_cast<const float4*>(in + i);
        uint2 u;
        u.x = pack_bf16x2(v.x * scale, v.y * scale);
        u.y = pack_bf16x2(v.z * scale, v.w * scale);
        *reinterpret_cast<uint2*>(out + i) = u;
    }
    if (i < n && i + 3 >= n)
        for (long long k = i; k < n; ++k) out[k] = __float2bfloat16_rn(in[k] * scale);
}

int f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, float scale, cudaStream_t s) {
    if (n <= 0) return 0;
    if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(out) & 7)) return set_error(ARD_ERR_SHAPE, "f32_to_bf16: unaligned");
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    f32_to_bf16_kernel<<<(unsigned)blocks, 256, 0, s>>>(in, out, n, scale);
    return check_cuda(cudaGetLastError(), "f32_to_bf16 launch");
}

__global__ void fill_f32_kernel(float* p, long long n, float v) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}
int fill_f32(float* p, long long n, float v, cudaStream_t s) {
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    fill_f32_kernel<<<(unsigned)blocks, 256, 0, s>>>(p, n, v);
    return check_cuda(cudaGetLastError(), "fill launch");
}

// quantize_tensor, src/residual.py:210-212: clamp(-1,1) * 32767 -> int16 (truncation toward zero) -> float / 32767
__global__ void quantize_kernel(const float* __restrict__ in, float* __restrict__ out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float c = fminf(fmaxf(in[i], -1.0f), 1.0f);
        out[i] = truncf(c * 32767.0f) / 32767.0f;
    }
}
int quantize_waveform(const float* in, float* out, long long n, cudaStream_t s) {
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    quantize_kernel<<<(unsigned)blocks, 256, 0, s>>>(in, out, n);
    return check_cuda(cudaGetLastError(), "quantize launch");
}

}  // namespace ard

// ================================================================================================ backward row-wise kernels
// (ResiDual training step, reference: loss.backward() in src/training.py:30-32 through the frozen encoder)
namespace ard {

// LayerNorm backward: y = (x - mean) * rstd * gamma + beta over the last dim C.
//   dx = rstd * (gg - mean(gg) - xhat * mean(gg * xhat)),  gg = g * gamma;   out = (add ? add : 0) + dx   (fp32)
// Rows may be the PatchMerging gather (MergeRows): x is read and dx written through the same row map.
//   out = add_scale * add + dx  (fp32);   out_bf = bf16(add + dx)  (optional: the next dgrad GEMM's A operand)
// EXT: out_bf = bf16(add + dx + ext), ext read at row r = clip * ext.T + t from ext.p + clip * ext.bstride + t * C (a block's rows of a
// layers_residuals gradient, which reaches the dgrad operand only, never the fp32 shortcut gradient `out`).
template <int VEC, int NV, class Rows, bool EXT = false>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(Rows xrows, Rows orows, float* __restrict__ out_base,
                                                           const float* __restrict__ g, const float* __restrict__ gamma,
                                                           const float* __restrict__ add, float add_scale,
                                                           __nv_bfloat16* __restrict__ out_bf, long long nrows, RowAddend ext = RowAddend()) {
    constexpr int C = 32 * VEC * NV;
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= nrows) return;
    float v[NV][VEC], gg[NV][VEC];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int e = (i * 32 + lane) * VEC;
        float gm[VEC];
        load_vec<VEC>(xrows.at(row, e), v[i]);
        load_vec<VEC>(g + row * C + e, gg[i]);
        load_vec<VEC>(gamma + e, gm);
#pragma unroll
        for (int k = 0; k < VEC; ++k) gg[i][k] *= gm[k];
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) s += v[i][k];
    const float mean = warp_sum(s) * (1.0f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            v[i][k] -= mean;
            q = fmaf(v[i][k], v[i][k], q);
        }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / C) + LN_EPS);
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            v[i][k] *= rstd;                 // xhat
            m1 += gg[i][k];
            m2 = fmaf(gg[i][k], v[i][k], m2);
        }
    m1 = warp_sum(m1) * (1.0f / C);
    m2 = warp_sum(m2) * (1.0f / C);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const int e = (i * 32 + lane) * VEC;
        float* op = out_base + (orows.at(row, e) - orows.x);
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            const float d = rstd * (gg[i][k] - m1 - v[i][k] * m2);
            const float a = add != nullptr ? add[op - out_base + k] : 0.f;
            op[k] = fmaf(add_scale, a, d);
            if constexpr (EXT) {
                out_bf[op - out_base + k] = __float2bfloat16_rn(a + d + ext.p[(row / ext.T) * ext.bstride + (row % ext.T) * C + e + k]);
            } else {
                if (out_bf != nullptr) out_bf[op - out_base + k] = __float2bfloat16_rn(a + d);
            }
        }
    }
}

template <class Rows>
static int launch_ln_bwd(Rows xr, Rows orr, float* out, const float* g, const float* gamma, const float* add, float add_scale,
                         __nv_bfloat16* out_bf, long long nrows, int C, cudaStream_t s, RowAddend ext = RowAddend()) {
    const int wpb = 8;
    const unsigned grid = (unsigned)((nrows + wpb - 1) / wpb);
    if (ext.p && !out_bf) return set_error(ARD_ERR_SHAPE, "layernorm_bwd: the addend goes to the bf16 copy only");
    ProfScope ps(PROF_LN, s, 16.0 * nrows * C, ((add ? 16.0 : 12.0) + (out_bf ? 2.0 : 0.0) + (ext.p ? 4.0 : 0.0)) * nrows * C);
#define ARD_LNB_CASE(c, vec, nv)                                                                                                           \
    case c:                                                                                                                                \
        if (ext.p) layernorm_bwd_kernel<vec, nv, Rows, true><<<grid, wpb * 32, 0, s>>>(xr, orr, out, g, gamma, add, add_scale, out_bf, nrows, ext); \
        else layernorm_bwd_kernel<vec, nv, Rows><<<grid, wpb * 32, 0, s>>>(xr, orr, out, g, gamma, add, add_scale, out_bf, nrows);         \
        break;
    switch (C) {
        ARD_LNB_CASE(96, 1, 3)
        ARD_LNB_CASE(128, 4, 1)
        ARD_LNB_CASE(192, 2, 3)
        ARD_LNB_CASE(256, 4, 2)
        ARD_LNB_CASE(384, 4, 3)
        ARD_LNB_CASE(512, 4, 4)
        ARD_LNB_CASE(768, 4, 6)
        ARD_LNB_CASE(1024, 4, 8)
        ARD_LNB_CASE(1536, 4, 12)
        ARD_LNB_CASE(2048, 4, 16)
        default: return set_error(ARD_ERR_SHAPE, "layernorm_bwd: unsupported width C=%d", C);
    }
#undef ARD_LNB_CASE
    return check_cuda(cudaGetLastError(), "layernorm_bwd launch");
}

int layernorm_bwd(const float* x, const float* g, const float* gamma, const float* add, float* out, long long rows, int C, cudaStream_t s,
                  float add_scale, __nv_bfloat16* out_bf, RowAddend ext) {
    if (rows <= 0) return 0;
    return launch_ln_bwd(PlainRows{x, C}, PlainRows{out, C}, out, g, gamma, add, add_scale, out_bf, rows, C, s, ext);
}

// PatchMerging backward of the gather + LayerNorm(4C): g [B*(H/2)*(W/2), 4C] -> dx [B, H*W, C] (every source element appears once)
int merge_layernorm_bwd(const float* x, const float* g, const float* gamma, float* dx, __nv_bfloat16* dx_bf, int B, int H, int W, int C,
                        cudaStream_t s) {
    const long long rows = (long long)B * (H / 2) * (W / 2);
    return launch_ln_bwd(MergeRows{x, H, W, C}, MergeRows{dx, H, W, C}, dx, g, gamma, nullptr, 1.0f, dx_bf, rows, 4 * C, s);
}

// dh <- dh * gelu'(hpre)   (both bf16 [n]); gelu'(x) = Phi(x) + x * phi(x)
__global__ void gelu_bwd_mul_kernel(__nv_bfloat16* __restrict__ dh, const __nv_bfloat16* __restrict__ hpre, long long n) {
    long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    const long long stride = (long long)gridDim.x * blockDim.x * 8;
    for (; i + 7 < n; i += stride) {
        uint4 a = *reinterpret_cast<const uint4*>(dh + i);
        const uint4 b = *reinterpret_cast<const uint4*>(hpre + i);
        __nv_bfloat162* ap = reinterpret_cast<__nv_bfloat162*>(&a);
        const __nv_bfloat162* bp = reinterpret_cast<const __nv_bfloat162*>(&b);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 d = __bfloat1622float2(ap[k]);
            const float2 x = __bfloat1622float2(bp[k]);
            const float p0 = gelu_erf_grad(x.x), p1 = gelu_erf_grad(x.y);
            d.x *= p0; d.y *= p1;
            ap[k] = __floats2bfloat162_rn(d.x, d.y);
        }
        *reinterpret_cast<uint4*>(dh + i) = a;
    }
}
int gelu_bwd_mul(__nv_bfloat16* dh, const __nv_bfloat16* hpre, long long n, cudaStream_t s) {
    if (n <= 0) return 0;
    if (n % 8) return set_error(ARD_ERR_SHAPE, "gelu_bwd_mul: n must be a multiple of 8");
    long long blocks = (n / 8 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    ProfScope ps(PROF_OTHER, s, 30.0 * n, 6.0 * n);
    gelu_bwd_mul_kernel<<<(unsigned)blocks, 256, 0, s>>>(dh, hpre, n);
    return check_cuda(cudaGetLastError(), "gelu_bwd_mul launch");
}

// Lambda gradient, reduced in-kernel (src/residual.py:39: x_scaled = x_proj * learnable):
//   dlam[k] += sum_t coef[t,k] * gcoef[t,k]  (k < K);   gsc[t,k] = bf16(gcoef[t,k] * lam[k])  (k < Kp: the gradient flowing on to x_proj)
// coef, gcoef fp32 [M, Kp]: rows are padded to Kp (a multiple of 16, the GEMMs' K granularity) while dlam holds only the K
// logical components. Each CTA reduces a slab of rows for 32 columns in registers/smem, one atomicAdd per column per CTA.
// SPLIT3 (fp32-grade backward): gsc is written in the split activation form [hi | hi | lo], [M, 3 Kp].
template <bool SPLIT3>
__global__ void __launch_bounds__(256) lambda_grad_kernel(const float* __restrict__ coef, const float* __restrict__ gcoef,
                                                         const float* __restrict__ lam, float* __restrict__ dlam,
                                                         __nv_bfloat16* __restrict__ gsc, long long M, int K, int Kp, long long rows_per_cta) {
    __shared__ float part[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + tx;
    const long long r0 = (long long)blockIdx.y * rows_per_cta, r1 = min(r0 + rows_per_cta, M);
    float acc = 0.f;
    if (col < Kp) {
        const float l = lam[col];
        for (long long r = r0 + ty; r < r1; r += 8) {
            const float c = coef[r * Kp + col], gc = gcoef[r * Kp + col];
            acc = fmaf(c, gc, acc);
            if constexpr (SPLIT3) {
                const float v = gc * l;
                const __nv_bfloat16 hi = __float2bfloat16_rn(v);
                __nv_bfloat16* o = gsc + r * 3LL * Kp + col;
                o[0] = hi;
                o[Kp] = hi;
                o[2 * Kp] = __float2bfloat16_rn(v - __bfloat162float(hi));
            } else {
                gsc[r * Kp + col] = __float2bfloat16_rn(gc * l);
            }
        }
    }
    part[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && col < K && dlam != nullptr) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += part[w][tx];
        atomicAdd(dlam + col, t);
    }
}
int lambda_grad(const float* coef, const float* gcoef, const float* lam, float* dlam, __nv_bfloat16* gsc, long long M, int K, int Kp,
                cudaStream_t s, bool split3) {
    if (M <= 0) return 0;
    const int cb = (Kp + 31) / 32;
    long long ysplit = (148 * 8) / cb + 1;
    long long rows_per_cta = (M + ysplit - 1) / ysplit;
    rows_per_cta = ((rows_per_cta + 7) / 8) * 8;
    ysplit = (M + rows_per_cta - 1) / rows_per_cta;
    ProfScope ps(PROF_OTHER, s, 3.0 * M * Kp, (split3 ? 14.0 : 10.0) * M * Kp);
    if (split3) lambda_grad_kernel<true><<<dim3(cb, (unsigned)ysplit), 256, 0, s>>>(coef, gcoef, lam, dlam, gsc, M, K, Kp, rows_per_cta);
    else lambda_grad_kernel<false><<<dim3(cb, (unsigned)ysplit), 256, 0, s>>>(coef, gcoef, lam, dlam, gsc, M, K, Kp, rows_per_cta);
    return check_cuda(cudaGetLastError(), "lambda_grad launch");
}

// out[b*T + t, c] = g[b, c] * scale   (token-mean backward, htsat.py:810-811)
__global__ void bcast_rows_kernel(const float* __restrict__ g, float* __restrict__ out, int B, int T, int C, float scale) {
    const long long total = (long long)B * T * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const long long b = i / ((long long)T * C);
        out[i] = g[b * C + c] * scale;
    }
}
int bcast_rows(const float* g, float* out, int B, int T, int C, float scale, cudaStream_t s) {
    bcast_rows_kernel<<<148 * 4, 256, 0, s>>>(g, out, B, T, C, scale);
    return check_cuda(cudaGetLastError(), "bcast_rows launch");
}

// y = a + b (fp32), optionally also a bf16 copy of the sum
__global__ void add_f32_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ y, __nv_bfloat16* __restrict__ ybf,
                               long long n) {
    long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const long long stride = (long long)gridDim.x * blockDim.x * 4;
    for (; i + 3 < n; i += stride) {
        float4 u = *reinterpret_cast<const float4*>(a + i);
        if (b != nullptr) {
            const float4 w = *reinterpret_cast<const float4*>(b + i);
            u.x += w.x; u.y += w.y; u.z += w.z; u.w += w.w;
        }
        if (y != nullptr) *reinterpret_cast<float4*>(y + i) = u;
        if (ybf != nullptr) {
            uint2 p;
            p.x = pack_bf16x2(u.x, u.y);
            p.y = pack_bf16x2(u.z, u.w);
            *reinterpret_cast<uint2*>(ybf + i) = p;
        }
    }
}
int add_f32(const float* a, const float* b, float* y, __nv_bfloat16* ybf, long long n, cudaStream_t s) {
    if (n <= 0) return 0;
    if (n % 4) return set_error(ARD_ERR_SHAPE, "add_f32: n must be a multiple of 4");
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    add_f32_kernel<<<(unsigned)blocks, 256, 0, s>>>(a, b, y, ybf, n);
    return check_cuda(cudaGetLastError(), "add_f32 launch");
}

}  // namespace ard
