// Eigenvalues of a batch of dense symmetric fp64 matrices (ard_sym_eigvals): the eigen-solve behind run_PCA's per-head spectra
// (src/analyze_attention.py:13-59), which only needs eigenvalues; and eigenvalues + eigenvectors (ard_sym_eigh: steps 1 and 2, then
// step 3) for compute_pca_components (src/residual.py:103-159) and run_PCA's per-head components.
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
//   3. eig_ql_kernel: implicit QL (tql2) on T, its rotations accumulated into Z_T = I; eig_rank_kernel: the ascending order;
//      eig_tfactor_kernel + eig_backtr_kernel: Z <- Q_B Z_T with the reflectors step 1 left below B's subdiagonal (dlarft / dlarfb);
//      eig_zout_kernel: sorted rows, exchange permutation undone.
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
constexpr int EIGH_MAX_D = 12288;  // ard_sym_eigh keeps T (2 D doubles) in shared memory

// per-matrix workspace (doubles): V [NB][D], W [NB][D], P [T][D] (SYMV partials), cc [T][2 NB] (per-strip dots), d [D], e [D],
// tau [D], e^2 [D], g [4]
struct Ws {
    long long D, T, per;
    long long oV, oW, oP, oC, oD, oE, oT, oE2, oG;
    __host__ __device__ explicit Ws(int D_) : D(D_), T((D_ + TS - 1) / TS) {
        oV = 0; oW = oV + NB * D; oP = oW + NB * D; oC = oP + T * D; oD = oC + 2 * NB * T; oE = oD + D; oT = oE + D; oE2 = oT + D;
        oG = oE2 + D;
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
// Householder reflector H = I - tau v v^T (v[j+1] = 1) and store v as V[jj]. v[j+2:] also goes back below the subdiagonal of B's
// column j (the LAPACK layout: nothing reads those entries again) and tau into its own slot, for ard_sym_eigh's back-transformation.
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
    for (int i = p + t; i < D; i += COLT) {
        if (i <= j + 1) { vrow[i] = i <= j ? 0.0 : 1.0; continue; }
        const double v = col[-i] * scal;
        vrow[i] = v;
        col[-i] = v;
    }
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

// d[D-1], Gershgorin interval [gl, gu], ||T|| and pivmin (dstebz); e^2 for the Sturm counts
__global__ void __launch_bounds__(256) eig_gersh_kernel(const double* __restrict__ A, long long stride, int D, double* __restrict__ ws,
                                                        long long wper) {
    __shared__ double red[8];
    const Ws L(D);
    double* wsb = ws + blockIdx.x * wper;
    double* d = wsb + L.oD;
    double* e = wsb + L.oE;
    double* e2 = e + 2 * L.D;                                  // oE2
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
    const double* e2 = wsb + L.oE2;
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

// ------------------------------------------------------------------------------------------------------- eigenvectors (ard_sym_eigh)
constexpr int QLT = 256;     // threads of eig_ql_kernel: one row of the rotation product per thread
constexpr int QLG = 8;       // QL sweeps applied per pass over Z_T
constexpr int BTM = 64;      // eigenvector rows per CTA of eig_backtr_kernel

// per-matrix workspace after Ws (doubles): Y [D][D] (row m = eigenvector m of T, then of B), Tf [npan][NB][NB] (dlarft T factors),
// lam [D] (QL eigenvalues), rank [D] (ints), rot [R][QLG][D][2] (each row-CTA's rotations of one pass)
struct EWs {
    long long oY, oTf, oLam, oRank, oRot, per;
    int R;
    __host__ __device__ static long long up(long long x) { return (x + 31) / 32 * 32; }    // 256-byte aligned (rot is read as double2)
    __host__ __device__ explicit EWs(int D) {
        const long long d = D, npan = (d - 1 + NB - 1) / NB;
        R = (D + QLT - 1) / QLT;
        oY = Ws(D).per; oTf = up(oY + d * d); oLam = up(oTf + npan * NB * NB); oRank = up(oLam + d); oRot = up(oRank + d);
        per = up(oRot + (long long)R * QLG * 2 * d);
    }
};

// Implicit QL with Wilkinson shifts (EISPACK tql2) on T = tridiag(e, d, e), accumulating the rotations into Z_T = I, stored as
// Y[i][k] = Z_T[k][i] so each eigenvector is a contiguous row and the threads that own consecutive rows k of Z_T read coalesced.
// CTA (x, b) owns rows [x QLT, x QLT + QLT) of matrix b's Z_T. Its thread 0 generates the rotations (serial, O(D) per sweep; every
// row-CTA of a matrix runs the same deterministic iteration on its own copy of T, so they need no inter-CTA sync), QLG sweeps at a
// time; then every thread applies those sweeps to its row in one pass over columns [bot, top], as a wavefront: sweep s trails
// sweep s-1 by one column and carries one value in a register. A pass reads and writes Z_T once per QLG sweeps.
// T is normalised by max(|d|, |e|) first (the rotations are scale-free; 1e+-20 inputs then converge under the same test).
// Convergence: |e[m]| <= eps * max_{l' <= l}(|d[l']| + |e[l']|) (tql2). At most 30 D sweeps per matrix (dsteqr's limit); past it
// info[b] = number of off-diagonals still above the test, else 0.
__global__ void __launch_bounds__(QLT) eig_ql_kernel(int D, double* __restrict__ ws, long long wper, int* __restrict__ info) {
    extern __shared__ double qsm[];
    __shared__ int lo_s[QLG], hi_s[QLG], ctl[2];
    __shared__ double red[QLT / 32];
    const EWs E(D);
    const Ws L(D);
    double* wsb = ws + blockIdx.y * wper;
    double* d = qsm;
    double* e = qsm + D;
    double* Y = wsb + E.oY;
    double* rot = wsb + E.oRot + (long long)blockIdx.x * QLG * 2 * D;
    const int t = threadIdx.x, k = blockIdx.x * QLT + t;
    double amax = 0.0;
    for (int i = t; i < D; i += QLT) {
        d[i] = wsb[L.oD + i];
        e[i] = i < D - 1 ? wsb[L.oE + i] : 0.0;
        amax = fmax(amax, fmax(fabs(d[i]), fabs(e[i])));
    }
    amax = block_max<QLT>(amax, red);
    if (amax > 0.0)
        for (int i = t; i < D; i += QLT) { d[i] /= amax; e[i] /= amax; }
    if (k < D)
        for (int i = 0; i < D; ++i) Y[(long long)i * D + k] = i == k ? 1.0 : 0.0;
    __syncthreads();
    // generator state (thread 0)
    int l = 0, it = 0, bad = 0;
    bool inblock = false;
    double f = 0.0, tst1 = 0.0;
    const int maxit = 30 * D;
    const double eps = DBL_EPSILON;
    for (;;) {
        if (t == 0) {
            int ns = 0;
            while (ns < QLG && l < D) {
                if (!inblock) tst1 = fmax(tst1, fabs(d[l]) + fabs(e[l]));
                int m = l;
                while (m < D - 1 && fabs(e[m]) > eps * tst1) ++m;
                if (m == l) {                                        // d[l] converged
                    d[l] += f;
                    e[l] = 0.0;
                    ++l;
                    inblock = false;
                    continue;
                }
                if (it >= maxit) {
                    for (int i = l; i < D - 1; ++i) bad += fabs(e[i]) > eps * tst1;
                    l = D;
                    break;
                }
                ++it;
                inblock = true;
                // one implicit QL sweep on [l, m]
                double g = d[l];
                double p = (d[l + 1] - g) / (2.0 * e[l]);
                double r = hypot(p, 1.0);
                if (p < 0) r = -r;
                d[l] = e[l] / (p + r);
                d[l + 1] = e[l] * (p + r);
                const double dl1 = d[l + 1];
                double h = g - d[l];
                for (int i = l + 2; i < D; ++i) d[i] -= h;
                f += h;
                p = d[m];
                double c = 1.0, c2 = 1.0, c3 = 1.0, s = 0.0, s2 = 0.0;
                const double el1 = e[l + 1];
                double* rs = rot + (long long)ns * 2 * D;
                for (int i = m - 1; i >= l; --i) {
                    c3 = c2; c2 = c; s2 = s;
                    g = c * e[i];
                    h = c * p;
                    r = hypot(p, e[i]);
                    e[i + 1] = s * r;
                    s = e[i] / r;
                    c = p / r;
                    p = c * d[i] - s * g;
                    d[i + 1] = h + s * (c * g + s * d[i]);
                    rs[2 * i] = c;
                    rs[2 * i + 1] = s;
                }
                p = -s * s2 * c3 * el1 * e[l] / dl1;
                e[l] = s * p;
                d[l] = c * p;
                lo_s[ns] = l;
                hi_s[ns] = m - 1;
                ++ns;
            }
            ctl[0] = ns;
            ctl[1] = l >= D;
        }
        __syncthreads();
        const int ns = ctl[0];
        if (ns > 0 && k < D) {
            int bot = D, top = 0, lo[QLG], hi[QLG];
            double hc[QLG];
#pragma unroll
            for (int q = 0; q < QLG; ++q) {
                lo[q] = q < ns ? lo_s[q] : D;                      // a sweep past ns is the identity
                hi[q] = q < ns ? hi_s[q] : -1;
                bot = min(bot, lo[q]);
                top = max(top, hi[q] + 1);
                hc[q] = 0.0;
            }
            // step i: sweep q consumes column i + q (sweep 0 reads it from Y) and hands column i + q + 1 on; the last one writes
            for (int i = top; i >= bot - QLG; --i) {
                double x = i >= bot ? Y[(long long)i * D + k] : 0.0;
                bool have = false;
#pragma unroll
                for (int q = 0; q < QLG; ++q) {
                    const int col = i + q;
                    if (col > top || col < bot - 1) { have = false; continue; }
                    if (col == top) { hc[q] = x; have = false; continue; }
                    if (col == bot - 1) { x = hc[q]; have = true; continue; }
                    double c = 1.0, sn = 0.0;
                    if (col >= lo[q] && col <= hi[q]) {
                        const double2 cs = *reinterpret_cast<const double2*>(rot + (long long)q * 2 * D + 2 * col);
                        c = cs.x;
                        sn = cs.y;
                    }
                    const double out = sn * x + c * hc[q];
                    hc[q] = c * x - sn * hc[q];
                    x = out;
                    have = true;
                }
                if (have) Y[(long long)(i + QLG) * D + k] = x;
            }
        }
        const bool done = ctl[1];
        __syncthreads();                                             // the rotations are consumed before thread 0 overwrites them
        if (done) break;
    }
    if (blockIdx.x == 0 && t == 0) info[blockIdx.y] = bad;
    if (blockIdx.x == 0)
        for (int i = t; i < D; i += QLT) wsb[E.oLam + i] = d[i];
}

// rank of eigenvalue m among the QL eigenvalues (ascending, ties by index): the row of Z it goes to
__global__ void __launch_bounds__(256) eig_rank_kernel(int D, double* __restrict__ ws, long long wper) {
    const int m = blockIdx.x * 256 + threadIdx.x;
    if (m >= D) return;
    const EWs E(D);
    double* wsb = ws + blockIdx.y * wper;
    const double* lam = wsb + E.oLam;
    const double x = lam[m];
    int r = 0;
    for (int j = 0; j < D; ++j) {
        const double y = lam[j];
        r += y < x || (y == x && j < m);
    }
    reinterpret_cast<int*>(wsb + E.oRank)[m] = r;
}

// dlarft (forward, columnwise) for every panel at once: CTA (P, b) forms G = V^T V of panel P's reflectors (read from below the
// subdiagonal of B, v[j+1] = 1) and T with Q_P = H_p ... H_{p+kb-1} = I - V T V^T: T[j][j] = tau_j, T[:j, j] = -tau_j T[:j, :j] G[:j, j].
__global__ void __launch_bounds__(NB * NB) eig_tfactor_kernel(const double* __restrict__ A, long long stride, int D,
                                                              double* __restrict__ ws, long long wper) {
    __shared__ double Vs[NB][NB + 1], G[NB][NB + 1], T[NB][NB + 1];
    const Ws L(D);
    const EWs E(D);
    const double* Ab = A + blockIdx.y * stride;
    double* wsb = ws + blockIdx.y * wper;
    const int P = blockIdx.x, p = P * NB, kb = min(NB, D - 1 - p), t = threadIdx.x, a = t >> 5, bcol = t & 31;
    double acc = 0.0;
    for (int i0 = p + 1; i0 < D; i0 += NB) {
        __syncthreads();
        {
            const int ii = t & 31, jj = t >> 5, i = i0 + ii, j = p + jj;
            Vs[ii][jj] = (jj < kb && i < D && i > j) ? (i == j + 1 ? 1.0 : Ab[baddr(D, i, j)]) : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int ii = 0; ii < NB; ++ii) acc += Vs[ii][a] * Vs[ii][bcol];
    }
    G[a][bcol] = acc;
    T[a][bcol] = 0.0;
    __syncthreads();
    if (t < 32) {
        for (int j = 0; j < kb; ++j) {
            const double tau = wsb[L.oT + p + j];
            double s = 0.0;
            if (t < j)
                for (int r = t; r < j; ++r) s += T[t][r] * G[r][j];
            __syncwarp();
            if (t < j) T[t][j] = -tau * s;
            if (t == 0) T[j][j] = tau;
            __syncwarp();
        }
    }
    __syncthreads();
    wsb[E.oTf + (long long)P * NB * NB + t] = T[a][bcol];
}

// Y <- Y Q_P^T = Y - (Y V) T^T V^T for panel P (applied last panel first, so that the rows of Y become Q_B z_m, Q_B = H_0 ... H_{D-2}).
// CTA (x, b) owns BTM rows of Y; V is read from below the subdiagonal of B in 32 x 32 tiles. fp64 FMA, 8 outputs per thread.
__global__ void __launch_bounds__(256) eig_backtr_kernel(const double* __restrict__ A, long long stride, int D, double* __restrict__ ws,
                                                         long long wper, int P) {
    __shared__ double Ys[BTM][NB + 1], Vs[NB][NB + 1], Ts[NB][NB + 1];
    const EWs E(D);
    const double* Ab = A + blockIdx.y * stride;
    double* wsb = ws + blockIdx.y * wper;
    double* Y = wsb + E.oY;
    const int p = P * NB, kb = min(NB, D - 1 - p), m0 = blockIdx.x * BTM, t = threadIdx.x, lane = t & 31, mg = t >> 5;
    for (int e = t; e < NB * NB; e += 256) Ts[e / NB][e % NB] = wsb[E.oTf + (long long)P * NB * NB + e];
    auto load_v = [&](int i0) {
        for (int e = t; e < NB * NB; e += 256) {
            const int ii = e & 31, jj = e >> 5, i = i0 + ii, j = p + jj;
            Vs[ii][jj] = (jj < kb && i < D && i > j) ? (i == j + 1 ? 1.0 : Ab[baddr(D, i, j)]) : 0.0;
        }
    };
    double acc[BTM / 8];
#pragma unroll
    for (int q = 0; q < BTM / 8; ++q) acc[q] = 0.0;
    for (int i0 = p + 1; i0 < D; i0 += NB) {               // W = Y V (rows m0.., thread: column lane, rows mg + 8 q)
        __syncthreads();
        load_v(i0);
        for (int e = t; e < BTM * NB; e += 256) {
            const int r = e >> 5, ii = e & 31, m = m0 + r, i = i0 + ii;
            Ys[r][ii] = (m < D && i < D) ? Y[(long long)m * D + i] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int ii = 0; ii < NB; ++ii) {
            const double v = Vs[ii][lane];
#pragma unroll
            for (int q = 0; q < BTM / 8; ++q) acc[q] += Ys[mg + 8 * q][ii] * v;
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < BTM / 8; ++q) Ys[mg + 8 * q][lane] = acc[q];    // W into the Y tile's storage
    __syncthreads();
#pragma unroll
    for (int q = 0; q < BTM / 8; ++q) {                    // W T^T (T upper triangular), back into the same storage
        double s = 0.0;
        for (int c = lane; c < NB; ++c) s += Ys[mg + 8 * q][c] * Ts[lane][c];
        acc[q] = s;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < BTM / 8; ++q) Ys[mg + 8 * q][lane] = acc[q];
    for (int i0 = p + 1; i0 < D; i0 += NB) {               // Y -= (W T^T) V^T (thread: column i0 + lane, rows mg + 8 q)
        __syncthreads();
        load_v(i0);
        __syncthreads();
        const int i = i0 + lane;
#pragma unroll
        for (int q = 0; q < BTM / 8; ++q) {
            const int r = mg + 8 * q, m = m0 + r;
            double s = 0.0;
#pragma unroll 8
            for (int jj = 0; jj < NB; ++jj) s += Ys[r][jj] * Vs[lane][jj];
            if (m < D && i < D) Y[(long long)m * D + i] -= s;
        }
    }
}

// Z[b][rank[m]][i] = Y[m][D-1-i]: ascending order, and A's eigenvector is J y (the reduction ran on B = J A J)
__global__ void __launch_bounds__(256) eig_zout_kernel(int D, const double* __restrict__ ws, long long wper, double* __restrict__ Z,
                                                       long long zstride) {
    const EWs E(D);
    const double* wsb = ws + blockIdx.y * wper;
    const int m = blockIdx.x;
    const double* y = wsb + E.oY + (long long)m * D;
    double* z = Z + blockIdx.y * zstride + (long long)reinterpret_cast<const int*>(wsb + E.oRank)[m] * D;
    for (int i = threadIdx.x; i < D; i += 256) z[i] = y[D - 1 - i];
}

}  // namespace

long long sym_eigvals_workspace(int D, int batch) {
    if (D < 1 || batch < 1) return 0;
    return Ws(D).per * (long long)batch * (long long)sizeof(double);
}

long long sym_eigh_workspace(int D, int batch) {
    if (D < 1 || batch < 1) return 0;
    return EWs(D).per * (long long)batch * (long long)sizeof(double);
}

namespace {

int check_args(const char* fn, const double* A, long long stride, int D, int batch, const double* w, const void* work) {
    if (D < 1 || batch < 1) return set_error(ARD_ERR_SHAPE, "%s: need D >= 1 and batch >= 1 (D=%d, batch=%d)", fn, D, batch);
    if (stride < (long long)D * D) return set_error(ARD_ERR_SHAPE, "%s: stride %lld < D*D = %lld", fn, stride, (long long)D * D);
    if (!A || !w || !work) return set_error(ARD_ERR_SHAPE, "%s: NULL pointer (A=%p, w=%p, work=%p)", fn, (void*)A, (void*)w, work);
    if (batch > 65535) return set_error(ARD_ERR_SHAPE, "%s: batch %d > 65535", fn, batch);
    return 0;
}

// Householder tridiagonalisation + bisection (the whole of ard_sym_eigvals; ard_sym_eigh continues from its workspace). Launches
// counted except the last, which the caller checks.
int tridiag_bisect(double* A, long long stride, int D, int batch, double* w, double* ws, long long wper, cudaStream_t s) {
    const unsigned T = (unsigned)Ws(D).T;
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
    return 0;
}

}  // namespace

int sym_eigvals(double* A, long long stride, int D, int batch, double* w, void* work, long long work_bytes, cudaStream_t s) {
    ARD_TRY(check_args("ard_sym_eigvals", A, stride, D, batch, w, work));
    const long long need = sym_eigvals_workspace(D, batch);
    if (work_bytes < need) return set_error(ARD_ERR_SHAPE, "ard_sym_eigvals: workspace of %lld bytes < %lld needed", work_bytes, need);
    ARD_TRY(tridiag_bisect(A, stride, D, batch, w, (double*)work, Ws(D).per, s));
    return check_cuda(cudaGetLastError(), "ard_sym_eigvals bisection launch");
}

int sym_eigh(double* A, long long stride, int D, int batch, double* w, double* Z, long long zstride, int* info, void* work,
             long long work_bytes, cudaStream_t s) {
    ARD_TRY(check_args("ard_sym_eigh", A, stride, D, batch, w, work));
    if (!Z || !info) return set_error(ARD_ERR_SHAPE, "ard_sym_eigh: NULL pointer (Z=%p, info=%p)", (void*)Z, (void*)info);
    if (zstride < (long long)D * D) return set_error(ARD_ERR_SHAPE, "ard_sym_eigh: zstride %lld < D*D = %lld", zstride, (long long)D * D);
    if (D > EIGH_MAX_D) return set_error(ARD_ERR_SHAPE, "ard_sym_eigh: D %d > %d", D, EIGH_MAX_D);
    const long long need = sym_eigh_workspace(D, batch);
    if (work_bytes < need) return set_error(ARD_ERR_SHAPE, "ard_sym_eigh: workspace of %lld bytes < %lld needed", work_bytes, need);
    const EWs E(D);
    double* ws = (double*)work;
    const long long wper = E.per;
    ARD_TRY(tridiag_bisect(A, stride, D, batch, w, ws, wper, s));
    ARD_TRY(check_cuda(cudaGetLastError(), "ard_sym_eigh bisection launch"));
    const int qsm = 2 * D * (int)sizeof(double);
    if (qsm > 48 * 1024)
        ARD_TRY(check_cuda(cudaFuncSetAttribute(eig_ql_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, qsm), "ard_sym_eigh smem"));
    eig_ql_kernel<<<dim3(E.R, batch), QLT, qsm, s>>>(D, ws, wper, info);
    eig_rank_kernel<<<dim3((D + 255) / 256, batch), 256, 0, s>>>(D, ws, wper);
    int launches = 2;
    const int npan = (D - 1 + NB - 1) / NB;
    if (npan > 0) {
        eig_tfactor_kernel<<<dim3(npan, batch), NB * NB, 0, s>>>(A, stride, D, ws, wper);
        ++launches;
        for (int P = npan - 1; P >= 0; --P) {
            eig_backtr_kernel<<<dim3((D + BTM - 1) / BTM, batch), 256, 0, s>>>(A, stride, D, ws, wper, P);
            ++launches;
        }
    }
    eig_zout_kernel<<<dim3(D, batch), 256, 0, s>>>(D, ws, wper, Z, zstride);
    count_launch(launches);
    return check_cuda(cudaGetLastError(), "ard_sym_eigh output launch");
}

}  // namespace ard

extern "C" long long ard_sym_eigvals_workspace(int D, int batch) { return ard::sym_eigvals_workspace(D, batch); }

extern "C" int ard_sym_eigvals(double* A, long long stride, int D, int batch, double* w, void* work, long long work_bytes, void* stream) {
    return ard::sym_eigvals(A, stride, D, batch, w, work, work_bytes, (cudaStream_t)stream);
}

extern "C" long long ard_sym_eigh_workspace(int D, int batch) { return ard::sym_eigh_workspace(D, batch); }

extern "C" int ard_sym_eigh(double* A, long long stride, int D, int batch, double* w, double* Z, long long zstride, int* info,
                            void* work, long long work_bytes, void* stream) {
    return ard::sym_eigh(A, stride, D, batch, w, Z, zstride, info, work, work_bytes, (cudaStream_t)stream);
}
