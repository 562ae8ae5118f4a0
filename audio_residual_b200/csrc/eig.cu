// Eigenvalues of a batch of dense symmetric fp64 matrices (ard_sym_eigvals): the eigen-solve behind run_PCA's per-head spectra
// (src/analyze_attention.py:13-59), which only needs eigenvalues.
//
//   1. Householder reduction to tridiagonal form, blocked as in LAPACK dsytrd / dlatrd (lower triangle, panels of NB columns).
//      Per panel column j:  eig_column_kernel   applies the panel's earlier reflectors to column j (A(:,j) -= V W(j,:)^T + W V(j,:)^T),
//                                               forms the reflector (dlarfg);
//                           eig_symv_kernel     y = A22 v over the lower triangle only (each element feeds y_r and y_c; one
//                                               64-column strip per CTA, deterministic per-strip partials instead of atomics),
//                                               and per-strip partials of the panel-correction dots V^T v, W^T v;
//                           eig_wcol_kernel     w = tau (y - W (V^T v) - V (W^T v)) - tau/2 (w^T v) v   (dlatrd).
//      After each panel:    eig_trailing_kernel A22 -= V W^T + W V^T on the lower tiles (fp64 FMA, 64 x 64 tile per CTA).
//   2. eig_bisect_kernel: eigenvalues of T = tridiag(e, d, e) by bisection on Sturm counts (dstebz / dlaebz), one thread per
//      (matrix, eigenvalue index), from Gershgorin bounds, pivots guarded by pivmin, to an absolute tolerance of 2 eps ||T||.
//
// Every launch covers the whole batch (blockIdx.y / .z = matrix), so the D dependent column steps are paid once per call, not once
// per matrix: 3 launches per column + 1 per panel + 2, all asynchronous on the caller's stream, no host synchronisation.
//
// Storage. The caller's matrix is row-major with its lower triangle filled. The reduction runs on B = J A J (J the exchange
// matrix; same eigenvalues), whose lower triangle is A's lower triangle read backwards: B[r][c] = A[D-1-c][D-1-r]. A column of B
// is then a contiguous run of memory, so the column kernels and the tile loads (lanes along r) are coalesced.
#include <float.h>

#include "ard_internal.h"

namespace ard {
namespace {

constexpr int NB = 32;       // panel width (columns per rank-2 NB trailing update)
constexpr int TS = 64;       // SYMV strip / trailing-update tile
constexpr int COLT = 512;    // threads of eig_column_kernel (one CTA per matrix)
constexpr int WCOLT = 1024;  // threads of eig_wcol_kernel (one CTA per matrix)

// per-matrix workspace (doubles): V [NB][D], W [NB][D], P [T][D] (SYMV partials), cc [T][2 NB] (per-strip dots), d [D], e [D],
// tau / e^2 [D], g [4]
struct Ws {
    long long D, T, per;
    long long oV, oW, oP, oC, oD, oE, oT, oG;
    __host__ __device__ explicit Ws(int D_) : D(D_), T((D_ + TS - 1) / TS) {
        oV = 0; oW = oV + NB * D; oP = oW + NB * D; oC = oP + T * D; oD = oC + 2 * NB * T; oE = oD + D; oT = oE + D; oG = oT + D;
        per = (oG + 4 + 31) / 32 * 32;
    }
};

__device__ __forceinline__ long long baddr(int D, int r, int c) {   // B[r][c] (r >= c) in the caller's row-major A
    return (long long)(D - 1 - c) * D + (D - 1 - r);
}

template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    for (int i = 0; i < NT / 32; ++i) s += red[i];
    return s;
}

template <int NT>
__device__ __forceinline__ double block_max(double v, double* red) {
    for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    for (int i = 0; i < NT / 32; ++i) s = fmax(s, red[i]);
    return s;
}

// Column j = p + jj of the panel starting at p: bring it up to date with the panel's reflectors 0..jj-1, reduce it with a
// Householder reflector H = I - tau v v^T (v[j+1] = 1) and store v as V[jj].
__global__ void __launch_bounds__(COLT) eig_column_kernel(double* __restrict__ A, long long stride, int D, double* __restrict__ ws,
                                                          long long wper, int p, int jj) {
    __shared__ double vj[NB], wj[NB], red[COLT / 32], sc[2];
    const Ws L(D);
    double* Ab = A + blockIdx.x * stride;
    double* wsb = ws + blockIdx.x * wper;
    double* V = wsb + L.oV;
    double* W = wsb + L.oW;
    const int j = p + jj, t = threadIdx.x;
    if (t < jj) { vj[t] = V[(long long)t * D + j]; wj[t] = W[(long long)t * D + j]; }
    __syncthreads();
    double* col = Ab + baddr(D, 0, j);     // B[r][j] = col[-r]
    double amax = 0.0;
    for (int i = j + t; i < D; i += COLT) {
        double a = col[-i];
#pragma unroll 4
        for (int k = 0; k < jj; ++k) a -= V[(long long)k * D + i] * wj[k] + W[(long long)k * D + i] * vj[k];
        col[-i] = a;
        if (i > j + 1) amax = fmax(amax, fabs(a));
    }
    amax = block_max<COLT>(amax, red);     // (its barriers also publish the updated column to the block)
    double ss = 0.0;
    if (amax > 0.0)
        for (int i = j + 2 + t; i < D; i += COLT) { const double a = col[-i] / amax; ss += a * a; }
    ss = block_sum<COLT>(ss, red);
    if (t == 0) {
        const double alpha = col[-(j + 1)], xnorm = amax * sqrt(ss);
        double tau = 0.0, beta = alpha, scal = 0.0;
        if (xnorm > 0.0) {                 // dlarfg
            beta = -copysign(hypot(alpha, xnorm), alpha);
            tau = (beta - alpha) / beta;
            scal = 1.0 / (alpha - beta);
        }
        wsb[L.oD + j] = col[-j];
        wsb[L.oE + j] = beta;
        wsb[L.oT + j] = tau;
        sc[0] = scal;
    }
    __syncthreads();
    const double scal = sc[0];
    double* vrow = V + (long long)jj * D;
    for (int i = p + t; i < D; i += COLT) vrow[i] = i <= j ? 0.0 : (i == j + 1 ? 1.0 : col[-i] * scal);
}

// y = A22 v, A22 = B[j+1:, j+1:] (lower triangle read once), and the strip's share of the dots V^T v, W^T v. CTA (J, b) owns the
// 64-column strip J: for every 64-row tile I >= J it adds B[r][c] v[c] into the row sums of tile I and B[r][c] v[r] (r > c) into
// the strip's own column sums. P[J][x] receives the strip's whole contribution to y[x] (x >= 64 J), so y[x] = sum_{J <= x / 64} P[J][x].
__global__ void __launch_bounds__(256) eig_symv_kernel(const double* __restrict__ A, long long stride, int D, double* __restrict__ ws,
                                                       long long wper, int p, int jj) {
    __shared__ double vc[TS], vr[TS], rsum[2][8][TS], dsum[TS];
    const Ws L(D);
    const int j = p + jj, J = blockIdx.x, c0 = J * TS;
    if (c0 + TS <= j + 1) return;                             // strip entirely outside A22
    const double* Ab = A + blockIdx.y * stride;
    double* wsb = ws + blockIdx.y * wper;
    const double* v = wsb + L.oV + (long long)jj * D;
    double* P = wsb + L.oP + (long long)J * D;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    if (t < TS) { const int c = c0 + t; vc[t] = (c > j && c < D) ? v[c] : 0.0; }
    __syncthreads();
    // the panel-correction dots over this strip's rows: cc[J][k] = V[k] . v, cc[J][NB + k] = W[k] . v (k < jj), one warp per dot
    for (int qd = warp; qd < 2 * jj; qd += 8) {
        const double* src = wsb + (qd < jj ? L.oV + (long long)qd * D : L.oW + (long long)(qd - jj) * D);
        const int xa = c0 + lane, xb = c0 + lane + 32;
        double s = (xa > j && xa < D ? src[xa] * vc[lane] : 0.0) + (xb > j && xb < D ? src[xb] * vc[lane + 32] : 0.0);
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) wsb[L.oC + 2 * NB * J + (qd < jj ? qd : NB + qd - jj)] = s;
    }
    double colacc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) colacc[q] = 0.0;
    int buf = 0;
    for (int I = J; I * TS < D; ++I, buf ^= 1) {
        const int r0 = I * TS;
        __syncthreads();                                      // vr of the previous tile is consumed
        if (t < TS) { const int r = r0 + t; vr[t] = (r > j && r < D) ? v[r] : 0.0; }
        __syncthreads();
        const int ra = r0 + lane, rb = r0 + lane + 32;
        double a0[8], a1[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int cl = warp + 8 * q, c = c0 + cl;
            const bool cok = c > j && c < D;
            a0[q] = (cok && ra < D && ra >= c) ? Ab[baddr(D, ra, c)] : 0.0;
            a1[q] = (cok && rb < D && rb >= c) ? Ab[baddr(D, rb, c)] : 0.0;
        }
        const double va = vr[lane], vb = vr[lane + 32];
        double ra_s = 0.0, rb_s = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int cl = warp + 8 * q, c = c0 + cl;
            ra_s += a0[q] * vc[cl];
            rb_s += a1[q] * vc[cl];
            colacc[q] += (ra > c ? a0[q] * va : 0.0) + (rb > c ? a1[q] * vb : 0.0);   // the diagonal counts once (row side)
        }
        rsum[buf][warp][lane] = ra_s;
        rsum[buf][warp][lane + 32] = rb_s;
        __syncthreads();
        if (t < TS) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) s += rsum[buf][w][t];
            if (I == J) dsum[t] = s;
            else if (r0 + t < D) P[r0 + t] = s;
        }
    }
    // strip's own columns: column sums (reduced over the warp's lanes) + the diagonal tile's row sums
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        double s = colacc[q];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        colacc[q] = s;
    }
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int cl = warp + 8 * q;
            if (c0 + cl < D) P[c0 + cl] = colacc[q] + dsum[cl];
        }
    }
}

// w = tau (y - W (V^T v) - V (W^T v));  w -= tau/2 (w . v) v  -> W[jj] (zero above row j+1)
__global__ void __launch_bounds__(WCOLT) eig_wcol_kernel(int D, double* __restrict__ ws, long long wper, int p, int jj) {
    __shared__ double c1[NB], c2[NB], red[WCOLT / 32];
    const Ws L(D);
    double* wsb = ws + blockIdx.x * wper;
    const double* V = wsb + L.oV;
    double* W = wsb + L.oW;
    const double* P = wsb + L.oP;
    const int j = p + jj, t = threadIdx.x, J0 = (j + 1) / TS;
    if (t < 2 * jj) {                                        // sum the strips' dots
        const int k = t < jj ? t : NB + t - jj;
        double s = 0.0;
        for (int J = J0; J < L.T; ++J) s += wsb[L.oC + 2 * NB * J + k];
        if (t < jj) c1[t] = s;
        else c2[t - jj] = s;
    }
    __syncthreads();
    const double tau = wsb[L.oT + j];
    const double* v = V + (long long)jj * D;
    double* w = W + (long long)jj * D;
    double dot = 0.0;
    for (int x = j + 1 + t; x < D; x += WCOLT) {
        double y = 0.0;
#pragma unroll 8
        for (int J = J0; J <= x / TS; ++J) y += P[(long long)J * D + x];
#pragma unroll 8
        for (int k = 0; k < jj; ++k) y -= W[(long long)k * D + x] * c1[k] + V[(long long)k * D + x] * c2[k];
        const double wx = tau * y;
        w[x] = wx;
        dot += wx * v[x];
    }
    dot = block_sum<WCOLT>(dot, red);
    const double alpha2 = -0.5 * tau * dot;
    for (int x = p + t; x < D; x += WCOLT) w[x] = x <= j ? 0.0 : w[x] + alpha2 * v[x];
}

// A22 -= V W^T + W V^T for rows / columns >= q (lower tiles; k < kb panel columns). 64 x 64 tile per CTA, 4 x 4 per thread.
__global__ void __launch_bounds__(256) eig_trailing_kernel(double* __restrict__ A, long long stride, int D, const double* __restrict__ ws,
                                                           long long wper, int q, int kb) {
    constexpr int KC = 16;
    __shared__ double Vr[KC][TS], Wr[KC][TS], Vc[KC][TS], Wc[KC][TS];
    const int I = blockIdx.x, Jt = blockIdx.y;
    if (Jt > I || (Jt + 1) * TS <= q) return;                   // upper tiles, and tiles whose columns are all < q (so are their rows)
    const Ws L(D);
    double* Ab = A + blockIdx.z * stride;
    const double* wsb = ws + blockIdx.z * wper;
    const double* V = wsb + L.oV;
    const double* W = wsb + L.oW;
    const int r0 = I * TS, c0 = Jt * TS, t = threadIdx.x, tr = t & 15, tc = t >> 4;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int k0 = 0; k0 < kb; k0 += KC) {
        __syncthreads();
        for (int e = t; e < KC * TS; e += 256) {
            const int k = e / TS, x = e % TS, kk = k0 + k;
            const bool kok = kk < kb;
            const int r = r0 + x, c = c0 + x;
            Vr[k][x] = (kok && r < D) ? V[(long long)kk * D + r] : 0.0;
            Wr[k][x] = (kok && r < D) ? W[(long long)kk * D + r] : 0.0;
            Vc[k][x] = (kok && c < D) ? V[(long long)kk * D + c] : 0.0;
            Wc[k][x] = (kok && c < D) ? W[(long long)kk * D + c] : 0.0;
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < KC; ++k) {
            double vr[4], wr[4], vc[4], wc[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) { vr[a] = Vr[k][tr + 16 * a]; wr[a] = Wr[k][tr + 16 * a]; }
#pragma unroll
            for (int b = 0; b < 4; ++b) { vc[b] = Vc[k][tc * 4 + b]; wc[b] = Wc[k][tc * 4 + b]; }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = fma(vr[a], wc[b], fma(wr[a], vc[b], acc[a][b]));
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int r = r0 + tr + 16 * a, c = c0 + tc * 4 + b;
            if (r < D && c >= q && r >= c) Ab[baddr(D, r, c)] -= acc[a][b];
        }
}

// d[D-1], Gershgorin interval [gl, gu], ||T|| and pivmin (dstebz); e^2 into the tau slot for the Sturm counts
__global__ void __launch_bounds__(256) eig_gersh_kernel(const double* __restrict__ A, long long stride, int D, double* __restrict__ ws,
                                                        long long wper) {
    __shared__ double red[8];
    const Ws L(D);
    double* wsb = ws + blockIdx.x * wper;
    double* d = wsb + L.oD;
    double* e = wsb + L.oE;
    double* e2 = wsb + L.oT;
    const int t = threadIdx.x;
    if (t == 0) d[D - 1] = A[blockIdx.x * stride];            // B[D-1][D-1] = A[0][0], final after the last trailing update
    __syncthreads();
    double lo = DBL_MAX, hi = -DBL_MAX, em = 0.0;
    for (int i = t; i < D; i += 256) {
        const double el = i > 0 ? fabs(e[i - 1]) : 0.0, er = i < D - 1 ? fabs(e[i]) : 0.0;
        lo = fmin(lo, d[i] - el - er);
        hi = fmax(hi, d[i] + el + er);
        if (i < D - 1) { em = fmax(em, er * er); e2[i] = e[i] * e[i]; }
    }
    const double glo = -block_max<256>(-lo, red);
    const double ghi = block_max<256>(hi, red);
    const double emax2 = block_max<256>(em, red);
    if (t == 0) {
        wsb[L.oG + 0] = glo;
        wsb[L.oG + 1] = ghi;
        wsb[L.oG + 2] = fmax(fabs(glo), fabs(ghi));
        wsb[L.oG + 3] = DBL_MIN * fmax(1.0, emax2);
    }
}

// eigenvalue m (ascending) of matrix b: bisection on the number of eigenvalues below x (Sturm sequence of T - x I)
__global__ void __launch_bounds__(128) eig_bisect_kernel(int D, const double* __restrict__ ws, long long wper, double* __restrict__ w) {
    const int m = blockIdx.x * 128 + threadIdx.x;
    if (m >= D) return;
    const Ws L(D);
    const double* wsb = ws + blockIdx.y * wper;
    const double* d = wsb + L.oD;
    const double* e2 = wsb + L.oT;
    const double tnorm = wsb[L.oG + 2], pivmin = wsb[L.oG + 3];
    double* out = w + (long long)blockIdx.y * D + m;
    if (tnorm == 0.0) { *out = 0.0; return; }
    const double eps = DBL_EPSILON * 0.5;                      // unit roundoff, as dlamch('P')
    double lo = wsb[L.oG + 0] - 2.1 * tnorm * eps * D - 4.2 * pivmin;
    double hi = wsb[L.oG + 1] + 2.1 * tnorm * eps * D + 4.2 * pivmin;
    const double atol = fmax(2.0 * DBL_EPSILON * tnorm, pivmin);
    for (int it = 0; it < 256 && hi - lo > atol; ++it) {
        const double x = 0.5 * (lo + hi);
        if (x <= lo || x >= hi) break;
        int cnt = 0;
        double qv = d[0] - x;
        if (fabs(qv) <= pivmin) qv = -pivmin;
        cnt += qv < 0.0;
        for (int i = 1; i < D; ++i) {
            qv = (d[i] - x) - e2[i - 1] / qv;
            if (fabs(qv) <= pivmin) qv = -pivmin;
            cnt += qv < 0.0;
        }
        if (cnt > m) hi = x;
        else lo = x;
    }
    *out = 0.5 * (lo + hi);
}

}  // namespace

long long sym_eigvals_workspace(int D, int batch) {
    if (D < 1 || batch < 1) return 0;
    return Ws(D).per * (long long)batch * (long long)sizeof(double);
}

int sym_eigvals(double* A, long long stride, int D, int batch, double* w, void* work, long long work_bytes, cudaStream_t s) {
    if (D < 1 || batch < 1) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: need D >= 1 and batch >= 1 (D=%d, batch=%d)", D, batch);
    if (stride < (long long)D * D) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: stride %lld < D*D = %lld", stride, (long long)D * D);
    if (!A || !w || !work) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: NULL pointer (A=%p, w=%p, work=%p)", (void*)A, (void*)w, work);
    const long long need = sym_eigvals_workspace(D, batch);
    if (work_bytes < need) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: workspace of %lld bytes < %lld needed", work_bytes, need);
    if (batch > 65535) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: batch %d > 65535", batch);
    const Ws L(D);
    double* ws = (double*)work;
    const long long wper = L.per;
    const unsigned T = (unsigned)L.T;
    int launches = 0;
    for (int p = 0; p < D - 1; p += NB) {
        const int kb = (D - 1 - p) < NB ? (D - 1 - p) : NB;
        for (int jj = 0; jj < kb; ++jj) {
            eig_column_kernel<<<batch, COLT, 0, s>>>(A, stride, D, ws, wper, p, jj);
            eig_symv_kernel<<<dim3(T, batch), 256, 0, s>>>(A, stride, D, ws, wper, p, jj);
            eig_wcol_kernel<<<batch, WCOLT, 0, s>>>(D, ws, wper, p, jj);
            launches += 3;
        }
        if (p + kb < D) {
            eig_trailing_kernel<<<dim3(T, T, batch), 256, 0, s>>>(A, stride, D, ws, wper, p + kb, kb);
            ++launches;
        }
        if (p == 0) ARD_TRY(check_cuda(cudaGetLastError(), "ard_sym_eigvals first panel launch"));
    }
    eig_gersh_kernel<<<batch, 256, 0, s>>>(A, stride, D, ws, wper);
    eig_bisect_kernel<<<dim3((D + 127) / 128, batch), 128, 0, s>>>(D, ws, wper, w);
    count_launch(launches);                                    // the two checked launches below and above count themselves
    return check_cuda(cudaGetLastError(), "ard_sym_eigvals bisection launch");
}

}  // namespace ard

extern "C" long long ard_sym_eigvals_workspace(int D, int batch) { return ard::sym_eigvals_workspace(D, batch); }

extern "C" int ard_sym_eigvals(double* A, long long stride, int D, int batch, double* w, void* work, long long work_bytes, void* stream) {
    return ard::sym_eigvals(A, stride, D, batch, w, work, work_bytes, (cudaStream_t)stream);
}
