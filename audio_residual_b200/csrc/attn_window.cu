// Shifted-window attention core for HTSAT (8x8 = 64-token windows, head_dim 24 or 32).
//
// Reference: WindowAttention.forward  CLAP/src/laion_clap/clap_module/htsat.py:326-352  (q k^T + relative-position bias
// + shift mask, softmax, attn @ v) together with the layout work SwinTransformerBlock.forward does around it
// (torch.roll / window_partition before, window_reverse / torch.roll after: htsat.py:452-474). Here the layout work
// costs nothing: qkv and the output both stay in TOKEN order in HBM and the cyclic shift + window gather/scatter is
// pure address arithmetic in this kernel's loads and stores (the proj Linear that follows is per-token, so it commutes
// with the permutation).
//
// One CTA (4 warps) per (clip, window, group of 2 heads; 2 measured faster than 4 or 1: more resident CTAs hide the gather). Each warp owns 16 query rows; the 64x64 score tile of one
// head lives entirely in registers (mma.sync m16n8k16 bf16 fragments), bias/mask/softmax are applied in registers and
// P feeds the second MMA directly from registers - S/P never touch shared or global memory unless the caller asks for
// the attention maps (`attn`, the block-mean capture of BasicLayer.forward htsat.py:589-595).
// The per-(window, head) problem is 64x64x24: far too small for a tcgen05 tile, and the kernel is bound by the softmax
// ALU/MUFU work (4096 exp per head-window vs 0.4 MFLOP of MMA), so the register-resident mma.sync form is the right tool.
#include <type_traits>

#include "ard_common.cuh"
#include "ard_internal.h"

namespace ard {

constexpr int AT_HEADS = 2;  // heads per CTA
constexpr int AT_TILE_BYTES = 3 * AT_HEADS * 64 * 64;
constexpr int AT_SMEM_BYTES = AT_TILE_BYTES + AT_HEADS * 232 * 4 + 2 * 64 * 4;

ARD_DEVINL void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
ARD_DEVINL void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
ARD_DEVINL void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
ARD_DEVINL void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
ARD_DEVINL void mma_bf16_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
ARD_DEVINL float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// smem tile of one head's Q, K or V: 64 rows x 64 bytes (head_dim padded to 32 bf16), 16-byte units XOR-swizzled by (row>>1)&3
ARD_DEVINL uint32_t tile_off(int row, int unit) { return (uint32_t)(row * 64 + ((unit ^ ((row >> 1) & 3)) << 4)); }

template <int HD>
__global__ void __launch_bounds__(128) window_attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                                                               const float* __restrict__ bias_table, float* __restrict__ attn,
                                                               float attn_scale, int attn_acc, int H, int W, int C, int nH, int shift) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int UPH = HD / 8;             // 16-byte units per head row (3 or 4)
    constexpr int UPR = AT_HEADS * UPH;     // units per (row, q|k|v) segment for this CTA's 4 heads
    constexpr int NT_O = HD / 8;            // output n-tiles
    extern __shared__ __align__(128) uint8_t dsm[];
    uint8_t* tiles = dsm;                                               // [part][head][64 rows][64 B]
    float (*tbl)[232] = reinterpret_cast<float (*)[232]>(dsm + AT_TILE_BYTES);
    int* tok_row = reinterpret_cast<int*>(dsm + AT_TILE_BYTES + AT_HEADS * 232 * 4);   // window token -> global row (b*T + token)
    int* tok_lab = tok_row + 64;                                        // shift-mask region label (htsat.py:414-437)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = nH / AT_HEADS;
    const int nWw = W >> 3, nW = (H >> 3) * nWw;
    const int g = blockIdx.x % G;
    const int wflat = blockIdx.x / G;       // b*nW + w
    const int w = wflat % nW;
    const long long b = wflat / nW;
    const int wh = w / nWw, ww = w % nWw;
    const int T = H * W;

    if (tid < 64) {
        const int th = tid >> 3, tw = tid & 7;
        const int hs = wh * 8 + th, ws = ww * 8 + tw;               // coordinates in the rolled image
        const int h = (hs + shift) % H, wd = (ws + shift) % W;      // torch.roll(x, -shift): rolled[hs] = x[(hs+shift)%H]
        tok_row[tid] = (int)(b * T + h * W + wd);
        int lab = 0;
        if (shift > 0) {
            const int rh = hs < H - 8 ? 0 : (hs < H - shift ? 1 : 2);
            const int rw = ws < W - 8 ? 0 : (ws < W - shift ? 1 : 2);
            lab = rh * 3 + rw;
        }
        tok_lab[tid] = lab;
    }
    static_assert(AT_HEADS == 2, "the bias-table load below fetches both heads of the CTA as one float2");
    for (int idx = tid; idx < 225; idx += 128) {    // nH is even, so the pair (idx, 2g), (idx, 2g+1) is 8-byte aligned
        const float2 bb = __ldg(reinterpret_cast<const float2*>(bias_table + idx * nH + g * AT_HEADS));
        tbl[0][idx] = bb.x;
        tbl[1][idx] = bb.y;
    }
    __syncthreads();

    // ---- gather q/k/v rows of this window (token order in HBM) into swizzled smem tiles
    // UPR consecutive threads copy the UPR 16-byte units of one (token, q|k|v) segment (coalesced 96 / 128-byte runs); the unit,
    // head and row-in-block indices are fixed per thread, so the 12 copies per thread need no index divisions (the kernel is
    // instruction-bound: the generic `i % UPR, i / UPR, ...` loop was ~45 % of a CTA's instructions together with the rest of
    // the prologue). 128 / UPR * UPR threads take part (96 of 128 for head_dim 24).
    {
        constexpr int TPB = 128 / UPR;               // tokens per pass (21 or 16)
        const int u = tid % UPR, tb = tid / UPR;
        const int hh = u / UPH, q = u - hh * UPH;
        if (tb < TPB) {
            const __nv_bfloat16* colp = qkv + (g * AT_HEADS) * HD + u * 8;
            uint8_t* dst0 = tiles + hh * 4096;
            for (int t = tb; t < 64; t += TPB) {
                const __nv_bfloat16* rowp = colp + (long long)tok_row[t] * (3 * C);
                const uint32_t off = tile_off(t, q);
#pragma unroll
                for (int part = 0; part < 3; ++part) cp_async16(dst0 + part * AT_HEADS * 4096 + off, rowp + part * C);
            }
        }
    }
    if constexpr (HD == 24) {  // zero the padded k-dim unit (unit 3) of every tile
        for (int i = tid; i < 3 * AT_HEADS * 64; i += 128) {
            const int t = i & 63, ph = i >> 6;
            *reinterpret_cast<uint4*>(tiles + ph * 4096 + tile_off(t, 3)) = make_uint4(0, 0, 0, 0);
        }
    }
    cp_async_wait_all();
    __syncthreads();

    const int r0 = warp * 16 + (lane >> 2);   // this thread's two query rows: r0 and r0 + 8
    const int ih0 = r0 >> 3, iw0 = r0 & 7, ih1 = ih0 + 1;
    // shift-mask bitmaps over this thread's 16 key columns
    uint32_t neq0 = 0, neq1 = 0;
    if (shift > 0 && (wh == (H >> 3) - 1 || ww == nWw - 1)) {
        const int l0 = tok_lab[r0], l1 = tok_lab[r0 + 8];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int lj = tok_lab[nt * 8 + (lane & 3) * 2 + e];
                neq0 |= (uint32_t)(lj != l0) << (nt * 2 + e);
                neq1 |= (uint32_t)(lj != l1) << (nt * 2 + e);
            }
    }
    const uint32_t tiles_u32 = smem_u32(tiles);
    constexpr float LOG2E = 1.4426950408889634f;

    // The shift mask is non-zero only in windows that straddle the roll seam (last window row / column of a shifted block): for
    // all other windows - every window of the unshifted blocks - the per-element mask test (LOP3 + ISETP + predicated FADD, a
    // quarter of the kernel's instructions, and the kernel is issue-bound at 77 % issue-active) is compiled out.
    const bool masked = shift > 0 && (wh == (H >> 3) - 1 || ww == nWw - 1);
    auto head_loop = [&](auto masked_tag) {
    constexpr bool MASKED = decltype(masked_tag)::value;
#pragma unroll 1
    for (int hh = 0; hh < AT_HEADS; ++hh) {
        const uint32_t qs = tiles_u32 + (0 * AT_HEADS + hh) * 4096;
        const uint32_t ks = tiles_u32 + (1 * AT_HEADS + hh) * 4096;
        const uint32_t vs = tiles_u32 + (2 * AT_HEADS + hh) * 4096;
        // Q fragments: 16 rows x 32 (padded) k
        uint32_t qa[2][4];
#pragma unroll
        for (int ksd = 0; ksd < 2; ++ksd)
            ldmatrix_x4(qs + tile_off(warp * 16 + (lane & 15), ksd * 2 + (lane >> 4)), qa[ksd][0], qa[ksd][1], qa[ksd][2], qa[ksd][3]);
        float s[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
            uint32_t kb0, kb1, kb2, kb3;
            ldmatrix_x4(ks + tile_off(nt * 8 + (lane & 7), lane >> 3), kb0, kb1, kb2, kb3);
            mma_bf16_16816(s[nt], qa[0][0], qa[0][1], qa[0][2], qa[0][3], kb0, kb1);
            mma_bf16_16816(s[nt], qa[1][0], qa[1][1], qa[1][2], qa[1][3], kb2, kb3);
        }
        // + relative position bias (htsat.py:337-340) + shift mask (htsat.py:342-345), row max
        float m0 = -INFINITY, m1 = -INFINITY;
        const float* tb = tbl[hh];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int jw = (lane & 3) * 2 + e;
                const int i0 = (ih0 - nt + 7) * 15 + (iw0 - jw + 7);
                float v0 = s[nt][e] + tb[i0];
                float v1 = s[nt][2 + e] + tb[i0 + 15];      // row r0+8: ih1 = ih0+1
                if constexpr (MASKED) {
                    if ((neq0 >> (nt * 2 + e)) & 1) v0 -= 100.0f;
                    if ((neq1 >> (nt * 2 + e)) & 1) v1 -= 100.0f;
                }
                s[nt][e] = v0;
                s[nt][2 + e] = v1;
                m0 = fmaxf(m0, v0);
                m1 = fmaxf(m1, v1);
            }
        (void)ih1;
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        const float mb0 = m0 * LOG2E, mb1 = m1 * LOG2E;
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const float p0 = ex2_approx(fmaf(s[nt][e], LOG2E, -mb0));
                const float p1 = ex2_approx(fmaf(s[nt][2 + e], LOG2E, -mb1));
                s[nt][e] = p0;
                s[nt][2 + e] = p1;
                sum0 += p0;
                sum1 += p1;
            }
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
        const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;

        if (attn != nullptr) {   // capture of the softmax probabilities (layers_attention)
            float* ap = attn + ((long long)wflat * nH + g * AT_HEADS + hh) * 4096;
            const float c0 = inv0 * attn_scale, c1 = inv1 * attn_scale;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                float2* d0 = reinterpret_cast<float2*>(ap + r0 * 64 + nt * 8 + (lane & 3) * 2);
                float2* d1 = reinterpret_cast<float2*>(ap + (r0 + 8) * 64 + nt * 8 + (lane & 3) * 2);
                float2 a = make_float2(s[nt][0] * c0, s[nt][1] * c0);
                float2 c = make_float2(s[nt][2] * c1, s[nt][3] * c1);
                if (attn_acc) {
                    const float2 o0 = *d0, o1 = *d1;
                    a.x += o0.x; a.y += o0.y; c.x += o1.x; c.y += o1.y;
                }
                *d0 = a;
                *d1 = c;
            }
        }

        // O = P V  (P from registers as the A operand)
        float o[NT_O][4];
#pragma unroll
        for (int nd = 0; nd < NT_O; ++nd) o[nd][0] = o[nd][1] = o[nd][2] = o[nd][3] = 0.f;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const uint32_t a0 = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
            const uint32_t a1 = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
            const uint32_t a2 = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            const uint32_t a3 = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
            const int krow = kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
#pragma unroll
            for (int np = 0; np < 2; ++np) {     // pairs of 8-wide output tiles: (0,1) and (2,3)
                uint32_t v0, v1, v2, v3;
                ldmatrix_x4_trans(vs + tile_off(krow, np * 2 + (lane >> 4)), v0, v1, v2, v3);
                mma_bf16_16816(o[np * 2], a0, a1, a2, a3, v0, v1);
                if (np * 2 + 1 < NT_O) mma_bf16_16816(o[(np * 2 + 1) < NT_O ? (np * 2 + 1) : 0], a0, a1, a2, a3, v2, v3);
            }
        }
        // normalise and park O (bf16) in this warp's own rows of the Q tile of head hh (nobody else reads them)
        uint8_t* qt = tiles + (0 * AT_HEADS + hh) * 4096;
#pragma unroll
        for (int nd = 0; nd < NT_O; ++nd) {
            *reinterpret_cast<uint32_t*>(qt + tile_off(r0, nd) + (lane & 3) * 4) = pack_bf16x2(o[nd][0] * inv0, o[nd][1] * inv0);
            *reinterpret_cast<uint32_t*>(qt + tile_off(r0 + 8, nd) + (lane & 3) * 4) = pack_bf16x2(o[nd][2] * inv1, o[nd][3] * inv1);
        }
    }
    };
    if (masked) head_loop(std::true_type{});
    else head_loop(std::false_type{});
    __syncwarp();
    // ---- scatter this warp's 16 output rows back to token order: (attn @ v).transpose(1,2).reshape(B_, N, C) htsat.py:354
    {   // UPR consecutive lanes store the UPR 16-byte units of one row (same division-free mapping as the gather)
        constexpr int RPP = 32 / UPR;                // rows per pass (5 or 4)
        const int u = lane % UPR, rb = lane / UPR;
        const int hh = u / UPH, q = u - hh * UPH;
        if (rb < RPP) {
            __nv_bfloat16* colp = out + (g * AT_HEADS) * HD + u * 8;
            const uint8_t* src0 = tiles + (0 * AT_HEADS + hh) * 4096;
            for (int r = rb; r < 16; r += RPP) {
                const int rr = warp * 16 + r;
                *reinterpret_cast<uint4*>(colp + (long long)tok_row[rr] * C) = *reinterpret_cast<const uint4*>(src0 + tile_off(rr, q));
            }
        }
    }
}

// ================================================================================================ backward
// Gradient of the window attention core w.r.t. q, k, v (token order, q pre-scaled), used by the ResiDual / probe training step
// (loss.backward() through the frozen encoder, src/training.py:30-32). Same CTA decomposition as the forward kernel: the
// probabilities are recomputed from the saved qkv (no S/P in HBM), and with P, dS in registers
//   dP = dO V^T,  delta = rowsum(dP . P),  dS = P . (dP - delta),  dQ = dS K        (per warp: its 16 query rows)
//   dV = P^T dO,  dK = dS^T Q                                                        (per warp: 16 KEY rows, P/dS via smem + ldmatrix.trans)
// GP: a probability gradient (ProbGrad) is added to dP before delta, read in the m16n8k16 accumulator layout of dp.
constexpr int ATB_TILE_BYTES = 4 * AT_HEADS * 64 * 64;            // q, k, v, dO
constexpr int ATB_PS_BYTES = 2 * 64 * 128;                        // P and dS of the head in flight (bf16 [64 q][64 keys])
constexpr int ATB_SMEM_BYTES = ATB_TILE_BYTES + ATB_PS_BYTES + AT_HEADS * 232 * 4 + 2 * 64 * 4;

ARD_DEVINL uint32_t ptile_off(int row, int unit) { return (uint32_t)(row * 128 + ((unit ^ (row & 7)) << 4)); }

template <int HD, bool GP = false>
__global__ void __launch_bounds__(128) window_attention_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout,
                                                                   __nv_bfloat16* __restrict__ dqkv, const float* __restrict__ bias_table,
                                                                   int H, int W, int C, int nH, int shift, ProbGrad<GP> pg = {}) {
    constexpr int UPH = HD / 8;
    constexpr int UPR = AT_HEADS * UPH;
    constexpr int NT_O = HD / 8;
    extern __shared__ __align__(128) uint8_t dsm[];
    uint8_t* tiles = dsm;                                               // [part 0..3][head][64 rows][64 B]
    uint8_t* ptile = dsm + ATB_TILE_BYTES;
    uint8_t* dstile = ptile + 64 * 128;
    float (*tbl)[232] = reinterpret_cast<float (*)[232]>(dsm + ATB_TILE_BYTES + ATB_PS_BYTES);
    int* tok_row = reinterpret_cast<int*>(dsm + ATB_TILE_BYTES + ATB_PS_BYTES + AT_HEADS * 232 * 4);
    int* tok_lab = tok_row + 64;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = nH / AT_HEADS;
    const int nWw = W >> 3, nW = (H >> 3) * nWw;
    const int g = blockIdx.x % G;
    const int wflat = blockIdx.x / G;
    const int w = wflat % nW;
    const long long b = wflat / nW;
    const int wh = w / nWw, ww = w % nWw;
    const int T = H * W;

    if (tid < 64) {
        const int th = tid >> 3, tw = tid & 7;
        const int hs = wh * 8 + th, ws = ww * 8 + tw;
        const int h = (hs + shift) % H, wd = (ws + shift) % W;
        tok_row[tid] = (int)(b * T + h * W + wd);
        int lab = 0;
        if (shift > 0) {
            const int rh = hs < H - 8 ? 0 : (hs < H - shift ? 1 : 2);
            const int rw = ws < W - 8 ? 0 : (ws < W - shift ? 1 : 2);
            lab = rh * 3 + rw;
        }
        tok_lab[tid] = lab;
    }
    for (int i = tid; i < AT_HEADS * 225; i += 128) {
        const int hh = i / 225, idx = i - hh * 225;
        tbl[hh][idx] = __ldg(bias_table + idx * nH + g * AT_HEADS + hh);
    }
    __syncthreads();

    for (int i = tid; i < 64 * 4 * UPR; i += 128) {
        const int u = i % UPR;
        const int rp = i / UPR;
        const int part = rp & 3, t = rp >> 2;
        const int hh = u / UPH, q = u - hh * UPH;
        const __nv_bfloat16* src = part < 3 ? qkv + (long long)tok_row[t] * (3 * C) + part * C + (g * AT_HEADS) * HD + u * 8
                                            : dout + (long long)tok_row[t] * C + (g * AT_HEADS) * HD + u * 8;
        cp_async16(tiles + (part * AT_HEADS + hh) * 4096 + tile_off(t, q), src);
    }
    if constexpr (HD == 24) {
        for (int i = tid; i < 4 * AT_HEADS * 64; i += 128) {
            const int t = i & 63, ph = i >> 6;
            *reinterpret_cast<uint4*>(tiles + ph * 4096 + tile_off(t, 3)) = make_uint4(0, 0, 0, 0);
        }
    }
    cp_async_wait_all();
    __syncthreads();

    const int r0 = warp * 16 + (lane >> 2);
    const int ih0 = r0 >> 3, iw0 = r0 & 7;
    uint32_t neq0 = 0, neq1 = 0;
    if (shift > 0) {
        const int l0 = tok_lab[r0], l1 = tok_lab[r0 + 8];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int lj = tok_lab[nt * 8 + (lane & 3) * 2 + e];
                neq0 |= (uint32_t)(lj != l0) << (nt * 2 + e);
                neq1 |= (uint32_t)(lj != l1) << (nt * 2 + e);
            }
    }
    const uint32_t tiles_u32 = smem_u32(tiles);
    const uint32_t pt_u32 = smem_u32(ptile), dst_u32 = smem_u32(dstile);
    constexpr float LOG2E = 1.4426950408889634f;

#pragma unroll 1
    for (int hh = 0; hh < AT_HEADS; ++hh) {
        const uint32_t qs = tiles_u32 + (0 * AT_HEADS + hh) * 4096;
        const uint32_t ks = tiles_u32 + (1 * AT_HEADS + hh) * 4096;
        const uint32_t vs = tiles_u32 + (2 * AT_HEADS + hh) * 4096;
        const uint32_t gs = tiles_u32 + (3 * AT_HEADS + hh) * 4096;
        uint32_t qa[2][4], ga[2][4];
#pragma unroll
        for (int ksd = 0; ksd < 2; ++ksd) {
            ldmatrix_x4(qs + tile_off(warp * 16 + (lane & 15), ksd * 2 + (lane >> 4)), qa[ksd][0], qa[ksd][1], qa[ksd][2], qa[ksd][3]);
            ldmatrix_x4(gs + tile_off(warp * 16 + (lane & 15), ksd * 2 + (lane >> 4)), ga[ksd][0], ga[ksd][1], ga[ksd][2], ga[ksd][3]);
        }
        float s[8][4], dp[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
            dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
            uint32_t b0, b1, b2, b3;
            ldmatrix_x4(ks + tile_off(nt * 8 + (lane & 7), lane >> 3), b0, b1, b2, b3);
            mma_bf16_16816(s[nt], qa[0][0], qa[0][1], qa[0][2], qa[0][3], b0, b1);
            mma_bf16_16816(s[nt], qa[1][0], qa[1][1], qa[1][2], qa[1][3], b2, b3);
            ldmatrix_x4(vs + tile_off(nt * 8 + (lane & 7), lane >> 3), b0, b1, b2, b3);
            mma_bf16_16816(dp[nt], ga[0][0], ga[0][1], ga[0][2], ga[0][3], b0, b1);
            mma_bf16_16816(dp[nt], ga[1][0], ga[1][1], ga[1][2], ga[1][3], b2, b3);
        }
        float m0 = -INFINITY, m1 = -INFINITY;
        const float* tb = tbl[hh];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int jw = (lane & 3) * 2 + e;
                const int i0 = (ih0 - nt + 7) * 15 + (iw0 - jw + 7);
                float v0 = s[nt][e] + tb[i0];
                float v1 = s[nt][2 + e] + tb[i0 + 15];
                if ((neq0 >> (nt * 2 + e)) & 1) v0 -= 100.0f;
                if ((neq1 >> (nt * 2 + e)) & 1) v1 -= 100.0f;
                s[nt][e] = v0;
                s[nt][2 + e] = v1;
                m0 = fmaxf(m0, v0);
                m1 = fmaxf(m1, v1);
            }
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        const float mb0 = m0 * LOG2E, mb1 = m1 * LOG2E;
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const float p0 = ex2_approx(fmaf(s[nt][e], LOG2E, -mb0));
                const float p1 = ex2_approx(fmaf(s[nt][2 + e], LOG2E, -mb1));
                s[nt][e] = p0;
                s[nt][2 + e] = p1;
                sum0 += p0;
                sum1 += p1;
            }
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
        sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
        sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
        const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;
        if constexpr (GP) {   // dp[nt][e]: query row r0, key nt*8 + (lane&3)*2 + e; dp[nt][2+e]: row r0 + 8
            const float* gp = pg.p + ((long long)wflat * nH + g * AT_HEADS + hh) * 4096 + r0 * 64 + (lane & 3) * 2;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float2 a = __ldg(reinterpret_cast<const float2*>(gp + nt * 8));
                const float2 c = __ldg(reinterpret_cast<const float2*>(gp + 8 * 64 + nt * 8));
                dp[nt][0] = fmaf(pg.scale, a.x, dp[nt][0]);
                dp[nt][1] = fmaf(pg.scale, a.y, dp[nt][1]);
                dp[nt][2] = fmaf(pg.scale, c.x, dp[nt][2]);
                dp[nt][3] = fmaf(pg.scale, c.y, dp[nt][3]);
            }
        }
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                s[nt][e] *= inv0;
                s[nt][2 + e] *= inv1;
                d0 = fmaf(s[nt][e], dp[nt][e], d0);
                d1 = fmaf(s[nt][2 + e], dp[nt][2 + e], d1);
            }
        d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
        d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
        d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
        d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
        // P and dS (bf16) to shared memory for the transposed products; dS stays in dp for dQ
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            dp[nt][0] = s[nt][0] * (dp[nt][0] - d0);
            dp[nt][1] = s[nt][1] * (dp[nt][1] - d0);
            dp[nt][2] = s[nt][2] * (dp[nt][2] - d1);
            dp[nt][3] = s[nt][3] * (dp[nt][3] - d1);
            *reinterpret_cast<uint32_t*>(ptile + ptile_off(r0, nt) + (lane & 3) * 4) = pack_bf16x2(s[nt][0], s[nt][1]);
            *reinterpret_cast<uint32_t*>(ptile + ptile_off(r0 + 8, nt) + (lane & 3) * 4) = pack_bf16x2(s[nt][2], s[nt][3]);
            *reinterpret_cast<uint32_t*>(dstile + ptile_off(r0, nt) + (lane & 3) * 4) = pack_bf16x2(dp[nt][0], dp[nt][1]);
            *reinterpret_cast<uint32_t*>(dstile + ptile_off(r0 + 8, nt) + (lane & 3) * 4) = pack_bf16x2(dp[nt][2], dp[nt][3]);
        }
        // dQ = dS K   (A = dS from registers, B = K read transposed, as V is in the forward's P V)
        float dq[NT_O][4], dk[NT_O][4], dv[NT_O][4];
#pragma unroll
        for (int nd = 0; nd < NT_O; ++nd) {
            dq[nd][0] = dq[nd][1] = dq[nd][2] = dq[nd][3] = 0.f;
            dk[nd][0] = dk[nd][1] = dk[nd][2] = dk[nd][3] = 0.f;
            dv[nd][0] = dv[nd][1] = dv[nd][2] = dv[nd][3] = 0.f;
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const uint32_t a0 = pack_bf16x2(dp[2 * kk][0], dp[2 * kk][1]);
            const uint32_t a1 = pack_bf16x2(dp[2 * kk][2], dp[2 * kk][3]);
            const uint32_t a2 = pack_bf16x2(dp[2 * kk + 1][0], dp[2 * kk + 1][1]);
            const uint32_t a3 = pack_bf16x2(dp[2 * kk + 1][2], dp[2 * kk + 1][3]);
            const int krow = kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
#pragma unroll
            for (int np = 0; np < 2; ++np) {
                uint32_t v0, v1, v2, v3;
                ldmatrix_x4_trans(ks + tile_off(krow, np * 2 + (lane >> 4)), v0, v1, v2, v3);
                mma_bf16_16816(dq[np * 2], a0, a1, a2, a3, v0, v1);
                if (np * 2 + 1 < NT_O) mma_bf16_16816(dq[(np * 2 + 1) < NT_O ? (np * 2 + 1) : 0], a0, a1, a2, a3, v2, v3);
            }
        }
        __syncthreads();   // P / dS tiles complete
        // dV = P^T dO, dK = dS^T Q for this warp's 16 KEY rows; A fragments come transposed out of the [q][key] tiles
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const int mi = lane >> 3;
            const int arow = kk * 16 + (mi >> 1) * 8 + (lane & 7);
            const int aunit = warp * 2 + (mi & 1);
            uint32_t p0, p1, p2, p3, e0, e1, e2, e3;
            ldmatrix_x4_trans(pt_u32 + ptile_off(arow, aunit), p0, p1, p2, p3);
            ldmatrix_x4_trans(dst_u32 + ptile_off(arow, aunit), e0, e1, e2, e3);
            const int krow = kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7);
#pragma unroll
            for (int np = 0; np < 2; ++np) {
                uint32_t v0, v1, v2, v3;
                ldmatrix_x4_trans(gs + tile_off(krow, np * 2 + (lane >> 4)), v0, v1, v2, v3);
                mma_bf16_16816(dv[np * 2], p0, p1, p2, p3, v0, v1);
                if (np * 2 + 1 < NT_O) mma_bf16_16816(dv[(np * 2 + 1) < NT_O ? (np * 2 + 1) : 0], p0, p1, p2, p3, v2, v3);
                ldmatrix_x4_trans(qs + tile_off(krow, np * 2 + (lane >> 4)), v0, v1, v2, v3);
                mma_bf16_16816(dk[np * 2], e0, e1, e2, e3, v0, v1);
                if (np * 2 + 1 < NT_O) mma_bf16_16816(dk[(np * 2 + 1) < NT_O ? (np * 2 + 1) : 0], e0, e1, e2, e3, v2, v3);
            }
        }
        __syncthreads();   // every warp is done reading this head's q/k/v/dO tiles and the P/dS tiles
        uint8_t* qt = tiles + (0 * AT_HEADS + hh) * 4096;
        uint8_t* kt = tiles + (1 * AT_HEADS + hh) * 4096;
        uint8_t* vt = tiles + (2 * AT_HEADS + hh) * 4096;
#pragma unroll
        for (int nd = 0; nd < NT_O; ++nd) {
            *reinterpret_cast<uint32_t*>(qt + tile_off(r0, nd) + (lane & 3) * 4) = pack_bf16x2(dq[nd][0], dq[nd][1]);
            *reinterpret_cast<uint32_t*>(qt + tile_off(r0 + 8, nd) + (lane & 3) * 4) = pack_bf16x2(dq[nd][2], dq[nd][3]);
            *reinterpret_cast<uint32_t*>(kt + tile_off(r0, nd) + (lane & 3) * 4) = pack_bf16x2(dk[nd][0], dk[nd][1]);
            *reinterpret_cast<uint32_t*>(kt + tile_off(r0 + 8, nd) + (lane & 3) * 4) = pack_bf16x2(dk[nd][2], dk[nd][3]);
            *reinterpret_cast<uint32_t*>(vt + tile_off(r0, nd) + (lane & 3) * 4) = pack_bf16x2(dv[nd][0], dv[nd][1]);
            *reinterpret_cast<uint32_t*>(vt + tile_off(r0 + 8, nd) + (lane & 3) * 4) = pack_bf16x2(dv[nd][2], dv[nd][3]);
        }
    }
    __syncwarp();
    // each warp parked dq/dk/dv for its own 16 rows: scatter them back to token order
    for (int i = lane; i < 16 * 3 * UPR; i += 32) {
        const int u = i % UPR;
        const int rp = i / UPR;
        const int part = rp % 3, rr = warp * 16 + rp / 3;
        const int hh = u / UPH, q = u - hh * UPH;
        const uint4 val = *reinterpret_cast<const uint4*>(tiles + (part * AT_HEADS + hh) * 4096 + tile_off(rr, q));
        *reinterpret_cast<uint4*>(dqkv + (long long)tok_row[rr] * (3 * C) + part * C + (g * AT_HEADS) * HD + u * 8) = val;
    }
}

int window_attention_bwd(const AttnArgs& a, const __nv_bfloat16* dout, __nv_bfloat16* dqkv, cudaStream_t s, const float* pgrad, float pscale) {
    if (a.B <= 0) return 0;
    if (a.nH <= 0 || a.C % a.nH != 0) return set_error(ARD_ERR_SHAPE, "window_attention_bwd: C=%d not divisible by heads=%d", a.C, a.nH);
    const int hd = a.C / a.nH;
    if ((a.H % 8) || (a.W % 8) || (a.nH % AT_HEADS)) return set_error(ARD_ERR_SHAPE, "window_attention_bwd: H=%d W=%d nH=%d unsupported", a.H, a.W, a.nH);
    int shift = a.shift;
    if (a.H <= 8 || a.W <= 8) shift = 0;
    const long long blocks = (long long)a.B * (a.H / 8) * (a.W / 8) * (a.nH / AT_HEADS);
    if (blocks > 0x7fffffffLL) return set_error(ARD_ERR_SHAPE, "window_attention_bwd: grid too large");
    static bool attr_set = false;
    if (!attr_set) {
        ARD_CUDA(cudaFuncSetAttribute(window_attention_bwd_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM_BYTES));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM_BYTES));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_bwd_kernel<24, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM_BYTES));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_bwd_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM_BYTES));
        attr_set = true;
    }
    const double tokens = (double)a.B * a.H * a.W;
    ProfScope ps(PROF_ATTN, s, 10.0 * tokens * 64 * a.C, tokens * a.C * 2.0 * 7.0 + (pgrad ? tokens * a.nH * 64 * 4.0 : 0.0));
    if (pgrad) {
        const ProbGrad<true> pg{pgrad, pscale};
        if (hd == 24)
            window_attention_bwd_kernel<24, true><<<(unsigned)blocks, 128, ATB_SMEM_BYTES, s>>>(a.qkv, dout, dqkv, a.bias_table, a.H, a.W, a.C, a.nH, shift, pg);
        else if (hd == 32)
            window_attention_bwd_kernel<32, true><<<(unsigned)blocks, 128, ATB_SMEM_BYTES, s>>>(a.qkv, dout, dqkv, a.bias_table, a.H, a.W, a.C, a.nH, shift, pg);
        else
            return set_error(ARD_ERR_SHAPE, "window_attention_bwd: head_dim %d unsupported (24 or 32)", hd);
        return check_cuda(cudaGetLastError(), "window_attention_bwd launch");
    }
    if (hd == 24)
        window_attention_bwd_kernel<24><<<(unsigned)blocks, 128, ATB_SMEM_BYTES, s>>>(a.qkv, dout, dqkv, a.bias_table, a.H, a.W, a.C, a.nH, shift);
    else if (hd == 32)
        window_attention_bwd_kernel<32><<<(unsigned)blocks, 128, ATB_SMEM_BYTES, s>>>(a.qkv, dout, dqkv, a.bias_table, a.H, a.W, a.C, a.nH, shift);
    else
        return set_error(ARD_ERR_SHAPE, "window_attention_bwd: head_dim %d unsupported (24 or 32)", hd);
    return check_cuda(cudaGetLastError(), "window_attention_bwd launch");
}

int window_attention(const AttnArgs& a, cudaStream_t s) {
    if (a.B <= 0) return 0;
    if (a.nH <= 0 || a.C % a.nH != 0) return set_error(ARD_ERR_SHAPE, "window_attention: C=%d not divisible by heads=%d", a.C, a.nH);
    const int hd = a.C / a.nH;
    if ((a.H % 8) || (a.W % 8) || (a.nH % AT_HEADS)) return set_error(ARD_ERR_SHAPE, "window_attention: H=%d W=%d nH=%d unsupported", a.H, a.W, a.nH);
    int shift = a.shift;
    if (a.H <= 8 || a.W <= 8) shift = 0;   // htsat.py:393-396
    const long long blocks = (long long)a.B * (a.H / 8) * (a.W / 8) * (a.nH / AT_HEADS);
    if (blocks > 0x7fffffffLL) return set_error(ARD_ERR_SHAPE, "window_attention: grid too large");
    static bool attr_set = false;
    if (!attr_set) {
        ARD_CUDA(cudaFuncSetAttribute(window_attention_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BYTES));
        ARD_CUDA(cudaFuncSetAttribute(window_attention_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BYTES));
        attr_set = true;
    }
    const double tokens = (double)a.B * a.H * a.W;
    ProfScope ps(PROF_ATTN, s, 4.0 * tokens * 64 * a.C, tokens * a.C * 2.0 * 4.0 + (a.attn_mean ? tokens * a.nH * 64 * 4.0 * (a.attn_accumulate ? 2 : 1) : 0.0));
    if (hd == 24)
        ARD_CUDA(enqueue_pdl(window_attention_kernel<24>, dim3((unsigned)blocks), dim3(128), AT_SMEM_BYTES, s, a.qkv, a.out, a.bias_table, a.attn_mean,
                            a.attn_scale, a.attn_accumulate, a.H, a.W, a.C, a.nH, shift));
    else if (hd == 32)
        ARD_CUDA(enqueue_pdl(window_attention_kernel<32>, dim3((unsigned)blocks), dim3(128), AT_SMEM_BYTES, s, a.qkv, a.out, a.bias_table, a.attn_mean,
                            a.attn_scale, a.attn_accumulate, a.H, a.W, a.C, a.nH, shift));
    else
        return set_error(ARD_ERR_SHAPE, "window_attention: head_dim %d unsupported (24 or 32)", hd);
    return check_cuda(cudaGetLastError(), "window_attention launch");
}

}  // namespace ard
