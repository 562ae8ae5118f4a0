// Small fp32 kernels around the encoder: audio_projection + L2 normalise (clap_module/model.py:539-543, :739-741),
// the ResiDual fold (src/residual.py:29-42 composed with WindowAttention.proj htsat.py:355), the token-semantic head
// (htsat.py:797-821) and the PCA moment accumulation (replaces IncrementalPCA.partial_fit, src/residual.py:137-138).
#include "ard_common.cuh"
#include "ard_internal.h"

namespace ard {

// ------------------------------------------------------------------------------------------------ small-batch Linear
// y[b, n] = act(sum_k x[b,k] W[n,k] + bias[n]);  one CTA = CL rows of x (held in smem) x a slice of the N outputs;
// one warp per output n, lanes stride over k (coalesced reads of W rows), CL accumulators per lane.
constexpr int LS_CL = 8;
__global__ void __launch_bounds__(256) linear_small_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ W,
                                                          const float* __restrict__ bias, float* __restrict__ y, int ldy, int B, int N,
                                                          int K, int act, int n_per_cta) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ float xs[];   // [LS_CL][K]
    const int b0 = blockIdx.y * LS_CL;
    const int nb = min(LS_CL, B - b0);
    for (int i = threadIdx.x; i < LS_CL * K; i += blockDim.x) {
        const int r = i / K, k = i - r * K;
        xs[i] = r < nb ? x[(long long)(b0 + r) * ldx + k] : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_begin = blockIdx.x * n_per_cta;
    const int n_end = min(n_begin + n_per_cta, N);
    for (int n = n_begin + warp; n < n_end; n += 8) {
        float acc[LS_CL];
#pragma unroll
        for (int r = 0; r < LS_CL; ++r) acc[r] = 0.f;
        const float* wr = W + (long long)n * K;
        if ((K & 3) == 0) {                           // 16-byte loads of the weight row and of the staged activations
            for (int k = lane * 4; k < K; k += 128) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(wr + k));
#pragma unroll
                for (int r = 0; r < LS_CL; ++r) {
                    const float4 xv = *reinterpret_cast<const float4*>(xs + r * K + k);
                    acc[r] = fmaf(w.x, xv.x, fmaf(w.y, xv.y, fmaf(w.z, xv.z, fmaf(w.w, xv.w, acc[r]))));
                }
            }
        } else {
            for (int k = lane; k < K; k += 32) {
                const float w = __ldg(wr + k);
#pragma unroll
                for (int r = 0; r < LS_CL; ++r) acc[r] = fmaf(w, xs[r * K + k], acc[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < LS_CL; ++r)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
        if (lane == 0) {
            const float bv = bias ? bias[n] : 0.f;
            for (int r = 0; r < nb; ++r) {
                float v = acc[r] + bv;
                if (act == ARD_ACT_RELU) v = fmaxf(v, 0.f);
                y[(long long)(b0 + r) * ldy + n] = v;
            }
        }
    }
}

int linear_small(const float* x, int ldx, const float* W, const float* bias, float* y, int ldy, int B, int N, int K, int act,
                 cudaStream_t s) {
    if (B <= 0) return 0;
    const int smem = LS_CL * K * 4;
    if (smem > 48 * 1024) return set_error(ARD_ERR_SHAPE, "linear_small: K=%d too large", K);
    const int n_per_cta = 64;
    dim3 grid((N + n_per_cta - 1) / n_per_cta, (B + LS_CL - 1) / LS_CL);
    ProfScope ps(PROF_HEAD, s, 2.0 * B * N * K, 4.0 * ((double)N * K + (double)B * K + (double)B * N));
    ARD_CUDA(enqueue_pdl(linear_small_kernel, grid, dim3(256), smem, s, x, ldx, W, bias, y, ldy, B, N, K, act, n_per_cta));
    return check_cuda(cudaGetLastError(), "linear_small launch");
}

// F.normalize(x, dim=-1): x / max(||x||_2, 1e-12); one warp per row
__global__ void l2_normalize_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int N) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= B) return;
    float s = 0.f;
    for (int k = lane; k < N; k += 32) {
        const float v = x[(long long)row * N + k];
        s = fmaf(v, v, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float inv = 1.0f / fmaxf(sqrtf(s), 1e-12f);
    for (int k = lane; k < N; k += 32) y[(long long)row * N + k] = x[(long long)row * N + k] * inv;
}

int l2_normalize(const float* x, float* y, int B, int N, cudaStream_t s) {
    if (B <= 0) return 0;
    ARD_CUDA(enqueue_pdl(l2_normalize_kernel, dim3((B + 7) / 8), dim3(256), 0, s, x, y, B, N));
    return check_cuda(cudaGetLastError(), "l2_normalize launch");
}

// backward of F.normalize: y = p / n, n = max(||p||, 1e-12):  dp = (g - y (y . g)) / n
__global__ void l2_normalize_bwd_kernel(const float* __restrict__ p, const float* __restrict__ g, float* __restrict__ out, int B, int N) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= B) return;
    float s = 0.f, d = 0.f;
    for (int k = lane; k < N; k += 32) {
        const float v = p[(long long)row * N + k];
        s = fmaf(v, v, s);
        d = fmaf(v, g[(long long)row * N + k], d);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        d += __shfl_xor_sync(0xffffffffu, d, o);
    }
    const float inv = 1.0f / fmaxf(sqrtf(s), 1e-12f);
    const float yg = d * inv;   // y . g
    for (int k = lane; k < N; k += 32) {
        const long long i = (long long)row * N + k;
        out[i] = (g[i] - p[i] * inv * yg) * inv;
    }
}
int l2_normalize_bwd(const float* p, const float* g, float* out, int B, int N, cudaStream_t s) {
    if (B <= 0) return 0;
    l2_normalize_bwd_kernel<<<(B + 7) / 8, 256, 0, s>>>(p, g, out, B, N);
    return check_cuda(cudaGetLastError(), "l2_normalize_bwd launch");
}

// g *= (act > 0)   (ReLU backward from the saved post-activation)
__global__ void relu_bwd_mul_kernel(float* __restrict__ g, const float* __restrict__ act, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        if (!(act[i] > 0.f)) g[i] = 0.f;
}
int relu_bwd_mul(float* g, const float* act, long long n, cudaStream_t s) {
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    relu_bwd_mul_kernel<<<(unsigned)blocks, 256, 0, s>>>(g, act, n);
    return check_cuda(cudaGetLastError(), "relu_bwd_mul launch");
}

// ------------------------------------------------------------------------------------------------ fp32 "TN" GEMM
// out_z[i][j] = sum_k a[k*lda + i] * (scale ? scale[k] : 1) * b_z[k*ldb + j];  i < Ma, j < Nb, z = blockIdx.z (up to 8 right-hand
// sides share `a`: the blocks of a layer share one ResiDual, so W'_b = M Wp_b for every block b is ONE launch).
// 64x64 tile, 4x4 per thread, 16-deep k-tiles double-buffered through registers (one __syncthreads per k-tile), 16-byte
// shared-memory reads. Only used to re-derive the folded ResiDual projection when lambda changes: C^3 flops per block, off the
// per-clip path, but once per training step - 3.6 GFLOP per step for HTSAT-tiny, all layers patched.
struct FoldBatch {
    const float* b[8];
    float* out_f32[8];          // either may be null
    __nv_bfloat16* out_bf16[8];
};
__global__ void __launch_bounds__(256) sgemm_tn_kernel(const float* __restrict__ a, int lda, FoldBatch fb, int ldb,
                                                      const float* __restrict__ scale, int ldo, int Ma, int Nb, int K) {
    __shared__ __align__(16) float As[2][16][64];
    __shared__ __align__(16) float Bs[2][16][64];
    const float* __restrict__ b = fb.b[blockIdx.z];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
    const int lk = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;   // this thread's float4 of a k-tile: row lk, columns lc..lc+3
    const bool a_ok = i0 + lc < Ma, b_ok = j0 + lc < Nb;            // Ma, Nb, lda, ldb are multiples of 4 (checked by the launcher)
    auto fetch = [&](int k0, float4& av, float4& bv) {
        const int k = k0 + lk;
        av = make_float4(0.f, 0.f, 0.f, 0.f);
        bv = av;
        if (k < K) {
            if (a_ok) {
                av = *reinterpret_cast<const float4*>(a + (long long)k * lda + i0 + lc);
                if (scale != nullptr) { const float sc = scale[k]; av.x *= sc; av.y *= sc; av.z *= sc; av.w *= sc; }
            }
            if (b_ok) bv = *reinterpret_cast<const float4*>(b + (long long)k * ldb + j0 + lc);
        }
    };
    float acc[4][4] = {};
    float4 av, bv;
    fetch(0, av, bv);
    *reinterpret_cast<float4*>(&As[0][lk][lc]) = av;
    *reinterpret_cast<float4*>(&Bs[0][lk][lc]) = bv;
    __syncthreads();
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += 16) {
        const bool more = k0 + 16 < K;
        if (more) fetch(k0 + 16, av, bv);
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
            const float ar[4] = {a4.x, a4.y, a4.z, a4.w}, br[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(ar[r], br[c], acc[r][c]);
        }
        if (more) {
            *reinterpret_cast<float4*>(&As[buf ^ 1][lk][lc]) = av;
            *reinterpret_cast<float4*>(&Bs[buf ^ 1][lk][lc]) = bv;
        }
        __syncthreads();
        buf ^= 1;
    }
    float* of = fb.out_f32[blockIdx.z];
    __nv_bfloat16* ob = fb.out_bf16[blockIdx.z];
    const int j = j0 + tx * 4;
    if (j >= Nb) return;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty * 4 + r;
        if (i >= Ma) break;
        if (of != nullptr) *reinterpret_cast<float4*>(of + (long long)i * ldo + j) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
        if (ob != nullptr) {
            uint2 pk;
            pk.x = pack_bf16x2(acc[r][0], acc[r][1]);
            pk.y = pack_bf16x2(acc[r][2], acc[r][3]);
            *reinterpret_cast<uint2*>(ob + (long long)i * ldo + j) = pk;
        }
    }
}

static int sgemm_tn(const float* a, int lda, const FoldBatch& fb, int nbatch, int ldb, const float* scale, int ldo, int Ma, int Nb, int K,
                    cudaStream_t s) {
    if ((Ma | Nb | lda | ldb | ldo) & 3) return set_error(ARD_ERR_SHAPE, "sgemm_tn: extents must be multiples of 4 (got %d x %d)", Ma, Nb);
    if (nbatch < 1 || nbatch > 8) return set_error(ARD_ERR_SHAPE, "sgemm_tn: batch of %d", nbatch);
    dim3 grid((Nb + 63) / 64, (Ma + 63) / 64, nbatch);
    ProfScope ps(PROF_OTHER, s, 2.0 * Ma * Nb * K * nbatch, 4.0 * ((double)Ma * K + ((double)Nb * K + (double)Ma * Nb) * nbatch));
    sgemm_tn_kernel<<<grid, 256, 0, s>>>(a, lda, fb, ldb, scale, ldo, Ma, Nb, K);
    return check_cuda(cudaGetLastError(), "sgemm_tn launch");
}

// b'_z[j] = sum_c d_z[c] M[c][j]   (the folded bias of up to 8 blocks sharing M): grid (C / 64, nbatch), 4 c-slices per column
struct FoldBiasBatch {
    const float* d[8];
    float* out[8];
};
__global__ void __launch_bounds__(256) fold_bias_kernel(FoldBiasBatch fb, const float* __restrict__ M, int C) {
    __shared__ float part[4][64];
    const float* __restrict__ d = fb.d[blockIdx.y];
    const int jj = threadIdx.x & 63, cs = threadIdx.x >> 6;
    const int j = blockIdx.x * 64 + jj;
    float acc = 0.f;
    if (j < C) {
#pragma unroll 4
        for (int c = cs; c < C; c += 4) acc = fmaf(d[c], M[(long long)c * C + j], acc);
    }
    part[cs][jj] = acc;
    __syncthreads();
    if (cs == 0 && j < C) fb.out[blockIdx.y][j] = (part[0][jj] + part[1][jj]) + (part[2][jj] + part[3][jj]);
}

// ResiDual (src/residual.py:37-42) applied to y = x Wp^T + bp:   r = ((y - mu) B^T * lambda) B = x (M Wp)^T + (bp - mu) M
// with M = B^T diag(lambda) B (symmetric).  Inputs: proj_w [C,C] fp32, dmean = bp - mu [C], basis [K,C], lam [K].
int residual_matrix(const float* basis, const float* lam, int C, int K, float* M, cudaStream_t s) {
    FoldBatch fb = {};
    fb.b[0] = basis; fb.out_f32[0] = M;
    return sgemm_tn(basis, C, fb, 1, C, lam, C, C, C, K, s);                         // M[i][j] = sum_k B[k][i] lam[k] B[k][j]
}
// One ResiDual shared by `nb` blocks of a layer (src/residual.py:170-186 builds one per layer): M once, then every block's
// W'_b = M Wp_b (fp32 and / or bf16 copies) and b'_b = (bp_b - mu) M in one launch each.
int residual_fold_batch(const float* const* proj_w, const float* const* dmean, const float* basis, const float* lam, int C, int K, float* Mtmp,
                        __nv_bfloat16* const* w_out, float* const* b_out, float* const* w_out_f32, int nb, cudaStream_t s) {
    if (nb < 1 || nb > 8) return set_error(ARD_ERR_SHAPE, "residual_fold_batch: %d blocks", nb);
    ARD_TRY(residual_matrix(basis, lam, C, K, Mtmp, s));
    FoldBatch fb = {};
    FoldBiasBatch bb = {};
    for (int z = 0; z < nb; ++z) {
        fb.b[z] = proj_w[z];
        fb.out_bf16[z] = w_out[z];
        fb.out_f32[z] = w_out_f32 ? w_out_f32[z] : nullptr;   // the fp32-grade mode splits the fp32 fold into bf16 terms
        bb.d[z] = dmean[z];
        bb.out[z] = b_out[z];
    }
    ARD_TRY(sgemm_tn(Mtmp, C, fb, nb, C, nullptr, C, C, C, C, s));                   // W'[i][j] = sum_c M[c][i] Wp[c][j]
    fold_bias_kernel<<<dim3((C + 63) / 64, nb), 256, 0, s>>>(bb, Mtmp, C);           // b'[j] = sum_c (bp-mu)[c] M[c][j]
    return check_cuda(cudaGetLastError(), "fold_bias launch");
}
int residual_fold(const float* proj_w, const float* dmean, const float* basis, const float* lam, int C, int K, float* Mtmp,
                  __nv_bfloat16* w_out, float* b_out, cudaStream_t s, float* w_out_f32) {
    return residual_fold_batch(&proj_w, &dmean, basis, lam, C, K, Mtmp, &w_out, &b_out, w_out_f32 ? &w_out_f32 : nullptr, 1, s);
}

// ------------------------------------------------------------------------------------------------ token-semantic head
// forward_features tail, htsat.py:798-821. normed [B, 64, C] (token = f*8 + t) is regrouped to x'[c][fb][g*8+t] with
// freq row f = g*2 + fb (4 time-quarters g stacked along frequency, 2 frequency bins each), then
//   fine_grained_embedding[b, 32*T' + r, c] = mean_fb x'[c][fb][T']                 (interpolate x32, utils.py:209-224)
//   y = Conv2d(C -> 527, kernel (2,3), padding (0,1))(x') -> [B, 527, 32]
//   framewise_output[b, 32*T' + r, o] = sigmoid(y[o][T']);  clipwise_output[b, o] = sigmoid(mean_T' y[o][T'])
// The conv is run as a GEMM over an im2col matrix A[(b,T'), (c, fb, kw)] (bf16) against tscam_conv.weight.view(527, 6C).
__global__ void tscam_im2col_kernel(const float* __restrict__ normed, __nv_bfloat16* __restrict__ A, int B, int C) {
    const long long total = (long long)B * 32 * C * 6;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int kw = (int)(i % 3);
        const int fb = (int)((i / 3) % 2);
        const int c = (int)((i / 6) % C);
        const long long row = i / (6LL * C);
        const int Tp = (int)(row % 32);
        const long long b = row / 32;
        const int tt = Tp + kw - 1;
        float v = 0.f;
        if (tt >= 0 && tt < 32) {
            const int gq = tt >> 3, t = tt & 7;
            const int f = gq * 2 + fb;
            v = normed[(b * 64 + f * 8 + t) * C + c];
        }
        A[i] = __float2bfloat16_rn(v);
    }
}

__global__ void tscam_finish_kernel(const float* __restrict__ y /*[B*32, ldy]*/, int ldy, float* __restrict__ framewise,
                                    float* __restrict__ clipwise, int B, int NC) {
    // one CTA per (clip); threads over classes
    const long long b = blockIdx.x;
    for (int o = threadIdx.x; o < NC; o += blockDim.x) {
        float s = 0.f;
        for (int Tp = 0; Tp < 32; ++Tp) {
            const float v = y[(b * 32 + Tp) * ldy + o];
            s += v;
            if (framewise) {
                const float sg = 1.0f / (1.0f + expf(-v));
                for (int r = 0; r < 32; ++r) framewise[(b * 1024 + Tp * 32 + r) * NC + o] = sg;
            }
        }
        if (clipwise) clipwise[b * NC + o] = 1.0f / (1.0f + expf(-s * (1.0f / 32.0f)));
    }
}

__global__ void fine_grained_kernel(const float* __restrict__ normed, float* __restrict__ fine, int B, int C) {
    const long long total = (long long)B * 1024 * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const int row = (int)((i / C) % 1024);
        const long long b = i / (1024LL * C);
        const int Tp = row >> 5;
        const int gq = Tp >> 3, t = Tp & 7;
        const float v0 = normed[(b * 64 + (gq * 2 + 0) * 8 + t) * C + c];
        const float v1 = normed[(b * 64 + (gq * 2 + 1) * 8 + t) * C + c];
        fine[i] = (v0 + v1) * 0.5f;
    }
}

// Backward of tscam_finish: dY[b*32 + T', o] = dL/dy[o][T'] from the pre-sigmoid y, for o < Kp (columns 527.. are zero, the
// K padding of the dgrad GEMM). Clipwise: g_clip * sigma'(mean y) / 32 (mean over the 32 steps); framewise: sigma'(y) times the
// sum of its 32 repeats (interpolate x32, utils.py:209-224). One CTA per (clip, T'), threads over classes. Output bf16 [rows, Kp]
// or, split3, the split activation form [hi | hi | lo] [rows, 3 Kp] of the fp32-grade dgrad.
__global__ void __launch_bounds__(256) tscam_bwd_dy_kernel(const float* __restrict__ y, int ldy, const float* __restrict__ g_frame,
                                                          const float* __restrict__ g_clip, __nv_bfloat16* __restrict__ dY, int Kp, int NC,
                                                          bool split3) {
    const long long row = blockIdx.x;
    const long long b = row / 32;
    const int Tp = (int)(row % 32);
    for (int o = threadIdx.x; o < Kp; o += blockDim.x) {
        float d = 0.f;
        if (o < NC) {
            if (g_clip) {
                float s = 0.f;
                for (int t = 0; t < 32; ++t) s += y[(b * 32 + t) * ldy + o];
                const float sg = 1.0f / (1.0f + expf(-s * (1.0f / 32.0f)));
                d = g_clip[b * NC + o] * sg * (1.0f - sg) * (1.0f / 32.0f);
            }
            if (g_frame) {
                const float sg = 1.0f / (1.0f + expf(-y[row * ldy + o]));
                float gs = 0.f;
                for (int r = 0; r < 32; ++r) gs += g_frame[(b * 1024 + Tp * 32 + r) * NC + o];
                d = fmaf(gs, sg * (1.0f - sg), d);
            }
        }
        const __nv_bfloat16 hi = __float2bfloat16_rn(d);
        if (split3) {
            __nv_bfloat16* r3 = dY + row * 3 * Kp;
            r3[o] = hi;
            r3[Kp + o] = hi;
            r3[2 * Kp + o] = __float2bfloat16_rn(d - __bfloat162float(hi));
        } else {
            dY[row * Kp + o] = hi;
        }
    }
}

// dL/d normed [B, 64, C] (token f*8 + t) = g_emb / 64 (token mean, htsat.py:810-811)
//   + col2im of dA [B*32, 6C] (the inverse of tscam_im2col_kernel: tokens (g*2 + fb)*8 + t feed column (c, fb, kw) of row T' = g*8+t-kw+1)
//   + g_fine summed over its 32 repeats / 2 (mean over the 2 frequency bins, htsat.py:807-808)
__global__ void tail_token_grad_kernel(const float* __restrict__ g_emb, const float* __restrict__ dA, const float* __restrict__ g_fine,
                                       float* __restrict__ out, int B, int C) {
    const long long total = (long long)B * 64 * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const int tok = (int)((i / C) % 64);
        const long long b = i / (64LL * C);
        const int f = tok >> 3, t = tok & 7, fb = f & 1;
        const int tt = (f >> 1) * 8 + t;
        float v = g_emb ? g_emb[b * C + c] * (1.0f / 64.0f) : 0.f;
        if (dA) {
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int Tp = tt - kw + 1;
                if (Tp >= 0 && Tp < 32) v += dA[(b * 32 + Tp) * 6LL * C + c * 6 + fb * 3 + kw];
            }
        }
        if (g_fine) {
            float s = 0.f;
            for (int r = 0; r < 32; ++r) s += g_fine[(b * 1024 + tt * 32 + r) * C + c];
            v = fmaf(0.5f, s, v);
        }
        out[i] = v;
    }
}

int tscam_bwd_dy(const float* y, int ldy, const float* g_frame, const float* g_clip, __nv_bfloat16* dY, int Kp, int B, bool split3,
                 cudaStream_t s) {
    ProfScope ps(PROF_HEAD, s, 0.0, 4.0 * B * 32 * ARD_CLASS_NUM * (1 + (g_clip ? 1 : 0) + (g_frame ? 33 : 0)));
    tscam_bwd_dy_kernel<<<B * 32, 256, 0, s>>>(y, ldy, g_frame, g_clip, dY, Kp, ARD_CLASS_NUM, split3);
    return check_cuda(cudaGetLastError(), "tscam_bwd_dy launch");
}
int tail_token_grad(const float* g_emb, const float* dA, const float* g_fine, float* out, int B, int C, cudaStream_t s) {
    ProfScope ps(PROF_HEAD, s, 0.0, 4.0 * B * 64 * C * (1 + (dA ? 3 : 0) + (g_fine ? 16 : 0)));
    tail_token_grad_kernel<<<148 * 8, 256, 0, s>>>(g_emb, dA, g_fine, out, B, C);
    return check_cuda(cudaGetLastError(), "tail_token_grad launch");
}

int tscam_im2col(const float* normed, __nv_bfloat16* A, int B, int C, cudaStream_t s) {
    tscam_im2col_kernel<<<148 * 8, 256, 0, s>>>(normed, A, B, C);
    return check_cuda(cudaGetLastError(), "tscam_im2col launch");
}
int tscam_finish(const float* y, int ldy, float* framewise, float* clipwise, int B, int NC, cudaStream_t s) {
    tscam_finish_kernel<<<B, 256, 0, s>>>(y, ldy, framewise, clipwise, B, NC);
    return check_cuda(cudaGetLastError(), "tscam_finish launch");
}
int fine_grained(const float* normed, float* fine, int B, int C, cudaStream_t s) {
    fine_grained_kernel<<<148 * 8, 256, 0, s>>>(normed, fine, B, C);
    return check_cuda(cudaGetLastError(), "fine_grained launch");
}

}  // namespace ard
