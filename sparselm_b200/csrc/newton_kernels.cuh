// Second-order phase of the batched solve (ill-conditioned pure-group problems, DESIGN section 2
// item 13): one lock-step damped Newton step on the active groups of k slow columns, entirely in
// this file's kernels -- Hessian assembly straight from the Gram, a batched blocked Cholesky
// factorisation H = U'U (64-wide panels: diagonal block factored and inverted in shared memory, the row
// panel through the inverse, trailing update on the FP64 tensor-core GEMM straight from those rows), blocked
// triangular solves, and the Armijo line search with objective differences formed without
// cancellation.  (Round 1 did these steps with torch operations and cuSOLVER's potrf.)
//
// On the active manifold of column c (groups with ||x_g|| > 0; identity on the other coordinates)
//     phi(x) = 1/(2n) x'Gx - c'x/n + sum_g w_g ||x_g|| + 1/2 sum_g d_g ||x_g||^2
//     grad   = (Gx - c)/n + w_g x_g/||x_g|| + d_g x_g
//     H      = G_AA/n + blockdiag_g( w_g/||x_g|| (I - u_g u_g') ) + diag(d),   u_g = x_g/||x_g||
// The system is factored on the ACTIVE coordinates only: column c has m_c of them (ACT[c][0..m_c), ascending),
// its matrix is the m_c x m_c compaction H[act][act] -- the factorisation costs sum_c m_c^3/3 instead of k p^3/3,
// and every kernel of the panel loop takes the per-column size from MS[c].
// Layouts: X, GX, U, KK, DP, GRAD, DIR are [k][ldv] (one row per column, solver feature order); ACT is
// [k][ldv] int; H is [k][ldh][ldh] row-major over the compacted coordinates (ldh from the largest m_c), upper
// triangle = the factor U after factorisation; group tables W2, D2, NRM are [k][Gn].
//
// Penalties with an l1 term (W1 [k][ldv] of per-coordinate l1 weights; NULL = pure group penalty): on the manifold
// where the signs s_j of the non-zero coordinates are fixed the objective gains the linear term sum_j w1_j s_j x_j,
//     grad += w1 * s   (no curvature: H is unchanged),
// and a coordinate is active iff x_j != 0 (a zero coordinate of an active group is inactive).  The line search
// starts from t0 = min(1, t_cross), t_cross = min{ -x_j/d_j : x_j d_j < 0 } the first sign change along the ray,
// so the l1 term stays linear over every tried step; a step accepted at t_cross stores the coordinates that reach
// zero as exact zeros (the support shrinks; it never grows here, that is the first-order iterations' job).
// Lasso has no group table: the caller passes one group of all p coordinates with zero weight.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

namespace slm {

constexpr int NW_NB = 64;   // panel width of the blocked Cholesky
constexpr int NW_T = 256;   // threads per block of the vector kernels
constexpr size_t NW_TILE_SMEM = 2 * NW_NB * (NW_NB + 1) * sizeof(double);  // two padded 64 x 64 tiles

__device__ __forceinline__ double nw_block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double t = (l < NW_T / 32) ? red[l] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}

__device__ __forceinline__ double nw_block_min(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double t = (l < NW_T / 32) ? red[l] : INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = fmin(t, __shfl_xor_sync(0xffffffffu, t, o));
    return t;
}

// step length at which coordinate j of x + t d reaches zero; +inf when it moves away from zero or stays
__device__ __forceinline__ double nw_cross(double xj, double dj) { return xj * dj < 0.0 ? -xj / dj : INFINITY; }

// u, kk, dp of one coordinate of a group with norm nrm, weight w, ridge d (kk = -1 marks an inactive coordinate)
__device__ __forceinline__ void nw_coord(long long e, double xj, double nrm, double w, double d, bool l1,
                                         double* __restrict__ U, double* __restrict__ KK, double* __restrict__ DP) {
    if (nrm > 0.0 && (!l1 || xj != 0.0)) {
        U[e] = xj / nrm;
        KK[e] = w / nrm;
        DP[e] = d;
    } else {
        U[e] = 0.0;
        KK[e] = -1.0;
        DP[e] = 0.0;
    }
}

// per column: group norms, activity, u = x/||x_g||, kk = w_g/||x_g||, dp = d_g (active coordinates); with l1
// weights (W1 != NULL) a zero coordinate is inactive even in an active group.  A single group with l1 weights
// (Lasso's zero-weight group of all p coordinates) is worked on by the whole block instead of one thread.
__global__ void __launch_bounds__(NW_T) newton_prepare_kernel(int p, int Gn, const int* __restrict__ gptr,
                                                              const double* __restrict__ X, long long ldv,
                                                              const double* __restrict__ W2, const double* __restrict__ D2,
                                                              const double* __restrict__ W1,
                                                              double* __restrict__ NRM, double* __restrict__ U,
                                                              double* __restrict__ KK, double* __restrict__ DP,
                                                              int* __restrict__ ACT, int* __restrict__ MS) {
    const int c = blockIdx.x;
    const double* x = X + (long long)c * ldv;
    __shared__ int wtot[NW_T / 32];
    __shared__ int base_s;
    __shared__ double red[NW_T / 32];
    const bool l1 = W1 != nullptr, whole = l1 && Gn == 1;
    if (whole) {
        const int ja = gptr[0], jb = gptr[1];
        double ss = 0.0;
        for (int j = ja + threadIdx.x; j < jb; j += NW_T) ss += x[j] * x[j];
        const double nrm = sqrt(nw_block_sum(ss, red));
        if (threadIdx.x == 0) NRM[c] = nrm;
        const double w = W2[c], d = D2 ? D2[c] : 0.0;
        for (int j = ja + threadIdx.x; j < jb; j += NW_T) nw_coord((long long)c * ldv + j, x[j], nrm, w, d, true, U, KK, DP);
    }
    for (int g = whole ? Gn : threadIdx.x; g < Gn; g += NW_T) {
        const int ja = gptr[g], jb = gptr[g + 1];
        double ss = 0.0;
        for (int j = ja; j < jb; ++j) ss += x[j] * x[j];
        const double nrm = sqrt(ss);
        NRM[(long long)c * Gn + g] = nrm;
        const double w = W2[(long long)c * Gn + g];
        const double d = D2 ? D2[(long long)c * Gn + g] : 0.0;
        for (int j = ja; j < jb; ++j) nw_coord((long long)c * ldv + j, x[j], nrm, w, d, l1, U, KK, DP);
    }
    // ordered list of the active coordinates (block-wide compaction, 256 coordinates per round)
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();  // also orders the KK writes above before the reads below
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j0 = 0; j0 < p; j0 += NW_T) {
        const int j = j0 + threadIdx.x;
        const bool on = j < p && KK[(long long)c * ldv + j] >= 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, on);
        if (lane == 0) wtot[warp] = __popc(bal);
        __syncthreads();
        int off = base_s, tot = 0;
#pragma unroll
        for (int w = 0; w < NW_T / 32; ++w) {
            if (w < warp) off += wtot[w];
            tot += wtot[w];
        }
        if (on) ACT[(long long)c * ldv + off + __popc(bal & ((1u << lane) - 1u))] = j;
        __syncthreads();
        if (threadIdx.x == 0) base_s += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) MS[c] = base_s;
}

// X[c][j] -> Z[fold[c]][j][slot[c]] (the Gram apply's feature-major layout; Z zero-filled by the caller)
__global__ void __launch_bounds__(NW_T) newton_pack_kernel(int p, const int* __restrict__ fold, const int* __restrict__ slot,
                                                           const double* __restrict__ X, long long ldv,
                                                           double* __restrict__ Z, long long ldz) {
    const int c = blockIdx.y;
    const int j = blockIdx.x * NW_T + threadIdx.x;
    if (j >= p) return;
    Z[((long long)fold[c] * p + j) * ldz + slot[c]] = X[(long long)c * ldv + j];
}

// gradient on the active coordinates from GX = G x:  grad = (Gx - c)/n + kk x + dp x  (kk x = w u), plus w1 sign(x)
// with l1 weights; gs (the quadratic part, stored in GS) is kept for the line search; GZ = G Z in the apply's layout
__global__ void __launch_bounds__(NW_T) newton_grad_kernel(int p, const double* __restrict__ G, long long g_stride,
                                                           long long pa, const int* __restrict__ fold,
                                                           const int* __restrict__ slot, const double* __restrict__ nobs,
                                                           const double* __restrict__ X, const double* __restrict__ GZ,
                                                           long long ldz, long long ldv, const double* __restrict__ KK,
                                                           const double* __restrict__ DP, const double* __restrict__ W1,
                                                           double* __restrict__ GS, double* __restrict__ GRAD) {
    const int c = blockIdx.y;
    const int j = blockIdx.x * NW_T + threadIdx.x;
    if (j >= p) return;
    const long long e = (long long)c * ldv + j;
    const double kk = KK[e];
    if (kk < 0.0) {
        GS[e] = 0.0;
        GRAD[e] = 0.0;
        return;
    }
    const double n = nobs[c];
    const double cj = G[(long long)fold[c] * g_stride + (long long)p * pa + j];
    const double gx = GZ[((long long)fold[c] * p + j) * ldz + slot[c]];  // (G x)_j in the apply's layout
    const double gs = (gx - cj) / n;
    GS[e] = gs;
    double g = gs + (kk + DP[e]) * X[e];
    if (W1) g += copysign(W1[e], X[e]);  // active: x_j != 0
    GRAD[e] = g;
}

// H[c][i][j] over the compacted coordinates i, j < m_c (original indices ACT[c][i], ACT[c][j]): the upper
// triangle and a band of 127 entries below the diagonal (the 128 x 128 diagonal tiles of the trailing updates
// are read whole); identity on the padding up to the next multiple of 8.
__global__ void __launch_bounds__(NW_T) newton_hessian_kernel(int p, const double* __restrict__ G, long long g_stride,
                                                              long long pa, const int* __restrict__ fold,
                                                              const double* __restrict__ nobs,
                                                              const int* __restrict__ gid, const double* __restrict__ U,
                                                              const double* __restrict__ KK, const double* __restrict__ DP,
                                                              long long ldv, const int* __restrict__ ACT,
                                                              const int* __restrict__ MS, double* __restrict__ H,
                                                              long long ldh) {
    const int c = blockIdx.z, i = blockIdx.y;
    const int j = blockIdx.x * NW_T + threadIdx.x;
    const int m = MS[c], mp = (m + 7) / 8 * 8;
    if (j >= mp || i >= mp || j < i - 127) return;  // the 128 x 128 diagonal tiles of the trailing updates start at any multiple of 64
    double* Hc = H + (long long)c * ldh * ldh;
    if (i >= m || j >= m) {  // padding rows / columns: identity
        Hc[(long long)i * ldh + j] = (i == j) ? 1.0 : 0.0;
        return;
    }
    const int oi = ACT[(long long)c * ldv + i], oj = ACT[(long long)c * ldv + j];
    const long long ei = (long long)c * ldv + oi, ej = (long long)c * ldv + oj;
    const double kki = KK[ei];
    double v = G[(long long)fold[c] * g_stride + (long long)oi * pa + oj] / nobs[c];
    if (gid[oi] == gid[oj]) v -= kki * U[ei] * U[ej];
    if (i == j) v += kki + DP[ei];
    Hc[(long long)i * ldh + j] = v;
}

// ---- blocked Cholesky, upper form H = U'U ------------------------------------------------------
// Working on the UPPER triangle of the row-major matrix keeps every bulk access on contiguous row
// segments: the panel to the right of a diagonal block is 64 full rows, and those rows ARE the
// K-major operands of the trailing update  H22 -= U12' U12  on the tensor-core GEMM (SYM, negate,
// upper tiles only: no transposed copies, no mirrored scattered stores).
//
// diagonal block [j0, j0+nb): factor in shared memory (A = U'U, U upper), write U back, invert it,
// keep the inverse in INV[c][panel][NB][NB] (row-major, upper triangular).  info[c] != 0: not
// positive definite.
//
// The 64 x 64 block is itself factored by 16-wide sub-blocks so that the kernel is not a chain of 64
// barrier-separated rank-1 steps: one warp factors a 16 x 16 diagonal sub-block in registers (row r in
// lane r, columns exchanged by shuffles; one rsqrt per pivot, no division), the rows below are solved
// against it one thread per row (forward substitution in registers), the rest is updated by the whole
// CTA (3 barriers per sub-block).  The four 16 x 16 inverses are then formed by four warps at once and
// the inverse of the 64 x 64 factor is assembled from them by block substitution.
constexpr int NW_SB = 16;
__global__ void __launch_bounds__(NW_T) chol_diag_kernel(double* __restrict__ H, long long ldh, int j0,
                                                         const int* __restrict__ MS, double* __restrict__ INV,
                                                         int npanels, int panel, int* __restrict__ info) {
    extern __shared__ double nw_sh[];
    double (*S)[NW_NB + 1] = reinterpret_cast<double (*)[NW_NB + 1]>(nw_sh);
    double (*V)[NW_NB + 1] = reinterpret_cast<double (*)[NW_NB + 1]>(nw_sh + NW_NB * (NW_NB + 1));
    constexpr int NSB = NW_NB / NW_SB;
    __shared__ double DI[NSB][NW_SB][NW_SB + 1];  // inverses of the diagonal sub-blocks (lower)
    __shared__ double TT[NSB - 1][NW_SB][NW_SB + 1];
    __shared__ double RD[NW_NB];  // reciprocals of the diagonal of L
    __shared__ int bad;
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = min(NW_NB, MS[c] - j0);
    if (nb <= 0) return;  // this column's matrix ended before the panel
    double* Hc = H + (long long)c * ldh * ldh + (long long)j0 * ldh + j0;
    if (tid == 0) bad = 0;
    // S holds the block TRANSPOSED (S[j][i] = A[i][j], i <= j): the factorisation below is the
    // familiar lower one on S, i.e. S = L = U'.  Identity beyond nb.
    for (int e = tid; e < NW_NB * NW_NB; e += NW_T) {
        const int i = e / NW_NB, j = e % NW_NB;  // consecutive threads: consecutive columns of a row (coalesced)
        S[j][i] = (i < nb && j < nb && i <= j) ? Hc[(long long)i * ldh + j] : (i == j ? 1.0 : 0.0);
        V[i][j] = 0.0;
    }
    __syncthreads();
    for (int kb = 0; kb < NSB; ++kb) {
        const int b0 = kb * NW_SB;
        if (warp == 0) {
            const int r = lane & (NW_SB - 1);  // lanes 16..31 mirror lanes 0..15 (their results are not stored)
            // entries right of the diagonal (q > r) are dead weight: never read by another lane, never stored --
            // the updates below run on them unconditionally, so the loop is free of per-lane branches
            double d[NW_SB];
#pragma unroll
            for (int q = 0; q < NW_SB; ++q) d[q] = S[b0 + r][b0 + q];
            bool ok = true;
            double myrs = 1.0;
#pragma unroll
            for (int k = 0; k < NW_SB; ++k) {
                const double piv = __shfl_sync(0xffffffffu, d[k], k);
                ok = ok && (piv > 0.0);
                const double rs = piv > 0.0 ? rsqrt(piv) : 1.0;
                d[k] *= rs;  // lane k: piv * rsqrt(piv) = sqrt(piv)
                myrs = (r == k) ? rs : myrs;
#pragma unroll
                for (int q = k + 1; q < NW_SB; ++q) {
                    const double lqk = __shfl_sync(0xffffffffu, d[k], q);
                    d[q] = fma(-d[k], lqk, d[q]);
                }
            }
            if (!ok && lane == 0) bad = 1;
            if (lane < NW_SB) {
#pragma unroll
                for (int q = 0; q < NW_SB; ++q)
                    if (q <= r) S[b0 + r][b0 + q] = d[q];
                RD[b0 + r] = myrs;
            }
        }
        __syncthreads();
        const int below = NW_NB - b0 - NW_SB;  // rows under the sub-block
        if (below > 0) {
            // rows below: L[r][b0 + q] by forward substitution against the sub-block, one thread per row
            if (tid < below) {
                const int r = b0 + NW_SB + tid;
                double a[NW_SB];
#pragma unroll
                for (int q = 0; q < NW_SB; ++q) a[q] = S[r][b0 + q];
#pragma unroll
                for (int m = 0; m < NW_SB; ++m) {
                    a[m] *= RD[b0 + m];
#pragma unroll
                    for (int q = m + 1; q < NW_SB; ++q) a[q] -= a[m] * S[b0 + q][b0 + m];
                }
#pragma unroll
                for (int q = 0; q < NW_SB; ++q) S[r][b0 + q] = a[q];
            }
            __syncthreads();
            // rest of the block: S[r][q] -= sum_m L[r][b0 + m] L[q][b0 + m]  (lower triangle, r >= q)
            for (int e = tid; e < below * below; e += NW_T) {
                const int r = b0 + NW_SB + e / below, q = b0 + NW_SB + e % below;
                if (q > r) continue;
                double a = 0.0;
#pragma unroll
                for (int m = 0; m < NW_SB; ++m) a += S[r][b0 + m] * S[q][b0 + m];
                S[r][q] -= a;
            }
            __syncthreads();
        }
    }
    for (int e = tid; e < nb * nb; e += NW_T) {
        const int i = e / nb, j = e % nb;
        if (i <= j) Hc[(long long)i * ldh + j] = S[j][i];  // U[i][j] = L[j][i]
    }
    // inverses of the four diagonal sub-blocks, one warp each: lane r forms column r of L_D^{-1} by forward
    // substitution, the rows of L_D come from the other lanes' registers
    if (warp < NSB) {
        const int b0 = warp * NW_SB, r = lane & (NW_SB - 1);
        double d[NW_SB], x[NW_SB];
#pragma unroll
        for (int q = 0; q < NW_SB; ++q) d[q] = S[b0 + r][b0 + q];
#pragma unroll
        for (int i = 0; i < NW_SB; ++i) {
            double acc = (i == r) ? 1.0 : 0.0;
#pragma unroll
            for (int m = 0; m < i; ++m) {
                const double lim = __shfl_sync(0xffffffffu, d[m], i);
                acc -= lim * x[m];  // x[m] = 0 for m < r
            }
            x[i] = (i >= r) ? acc * RD[b0 + i] : 0.0;
        }
        if (lane < NW_SB) {
#pragma unroll
            for (int i = 0; i < NW_SB; ++i) DI[warp][i][r] = x[i];
        }
    }
    __syncthreads();
    // V = L^{-1} (lower) by blocks: V_ii = DI_i, V_ij = -DI_i sum_{j <= m < i} L_im V_mj, by distance i - j
    {
        const int a = tid / NW_SB, b = tid % NW_SB;  // 256 threads = one 16 x 16 block
        for (int i = 0; i < NSB; ++i) V[i * NW_SB + a][i * NW_SB + b] = DI[i][a][b];
        __syncthreads();
        for (int dist = 1; dist < NSB; ++dist) {
            for (int j = 0; j + dist < NSB; ++j) {
                const int i = j + dist;
                double t = 0.0;
                for (int m = j; m < i; ++m)
#pragma unroll
                    for (int q = 0; q < NW_SB; ++q) t += S[i * NW_SB + a][m * NW_SB + q] * V[m * NW_SB + q][j * NW_SB + b];
                TT[j][a][b] = t;
            }
            __syncthreads();
            for (int j = 0; j + dist < NSB; ++j) {
                const int i = j + dist;
                double v = 0.0;
#pragma unroll
                for (int q = 0; q < NW_SB; ++q) v += DI[i][a][q] * TT[j][q][b];
                V[i * NW_SB + a][j * NW_SB + b] = -v;
            }
            __syncthreads();
        }
    }
    // stored as U^{-1} (upper): INV[i][j] = V[j][i]
    double* out = INV + ((long long)c * npanels + panel) * NW_NB * NW_NB;
    for (int e = tid; e < NW_NB * NW_NB; e += NW_T) out[e] = V[e % NW_NB][e / NW_NB];
    if (tid == 0 && bad) info[c] = 1;
}

// panel to the right of the diagonal block, in place: U12 = U11^{-T} A12, i.e.
// out[q][x] = sum_{m <= q} inv[m][q] A[m][x]  (inv = U11^{-1}, upper).  One block per 64 columns.
__global__ void __launch_bounds__(NW_T) chol_panel_kernel(double* __restrict__ H, long long ldh, int j0,
                                                          const int* __restrict__ MS, const double* __restrict__ INV,
                                                          int npanels, int panel) {
    extern __shared__ double nw_sh[];
    double (*A)[NW_NB + 1] = reinterpret_cast<double (*)[NW_NB + 1]>(nw_sh);
    double (*Vi)[NW_NB + 1] = reinterpret_cast<double (*)[NW_NB + 1]>(nw_sh + NW_NB * (NW_NB + 1));
    const int c = blockIdx.y, tid = threadIdx.x;
    const int p = MS[c];
    const int nb = min(NW_NB, p - j0);
    if (nb <= 0) return;
    const int x0 = j0 + nb + blockIdx.x * NW_NB;  // first column of this tile
    if (x0 >= p) return;
    const int nx = min(NW_NB, p - x0);
    double* Hc = H + (long long)c * ldh * ldh;
    const double* inv = INV + ((long long)c * npanels + panel) * NW_NB * NW_NB;
    for (int e = tid; e < NW_NB * NW_NB; e += NW_T) {
        const int m = e / NW_NB, x = e % NW_NB;  // rows of the panel are contiguous: coalesced
        A[m][x] = (m < nb && x < nx) ? Hc[(long long)(j0 + m) * ldh + x0 + x] : 0.0;
        Vi[m][x] = inv[e];
    }
    __syncthreads();
    for (int e = tid; e < NW_NB * NW_NB; e += NW_T) {
        const int q = e / NW_NB, x = e % NW_NB;
        if (q >= nb || x >= nx) continue;
        double a = 0.0;
        for (int m = 0; m <= q; ++m) a += Vi[m][q] * A[m][x];
        Hc[(long long)(j0 + q) * ldh + x0 + x] = a;
    }
}

// solve U'U d = rhs for every column with the blocked factor: forward (U'y = rhs) and backward (U d = y)
// substitution by panels; the diagonal blocks through their stored inverses.  rhs = -GRAD on the active
// coordinates; DIR receives d scattered back (inactive coordinates: 0).  A warp reads contiguous row segments
// of the factor (lanes over columns), partial sums meet in shared memory.  One block of NW_TS threads per
// column: the kernel streams m_c^2 x 8 bytes of the factor per column and is bound by the loads one block
// keeps in flight.
constexpr int NW_TS = 1024;
__global__ void __launch_bounds__(NW_TS) chol_solve_kernel(const double* __restrict__ H, long long ldh, int pfull,
                                                           const int* __restrict__ ACT, const int* __restrict__ MS,
                                                           const double* __restrict__ INV, int npanels,
                                                           const double* __restrict__ GRAD, double* __restrict__ DIR,
                                                           long long ldv) {
    extern __shared__ double sh[];  // y[ldh] + t[NB] + part[NWARP][NB]
    double* y = sh;
    double* t = sh + ldh;
    double* part = t + NW_NB;
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NWARP = NW_TS / 32;
    const int p = MS[c];
    const int* act = ACT + (long long)c * ldv;
    const double* Hc = H + (long long)c * ldh * ldh;
    for (int j = tid; j < pfull; j += NW_TS) DIR[(long long)c * ldv + j] = 0.0;
    for (int j = tid; j < p; j += NW_TS) y[j] = -GRAD[(long long)c * ldv + act[j]];
    __syncthreads();
    const int np = (p + NW_NB - 1) / NW_NB;
    // forward: y_j = U_jj^{-T} (rhs_j - sum_{i < j} U[i-rows][j-cols]' y_i)
    for (int pn = 0; pn < np; ++pn) {
        const int j0 = pn * NW_NB, nb = min(NW_NB, p - j0);
        double a0 = 0.0, a1 = 0.0;  // columns j0 + lane, j0 + lane + 32
        for (int i = warp; i < j0; i += NWARP) {
            const double* row = Hc + (long long)i * ldh + j0;
            const double yi = y[i];
            if (lane < nb) a0 += row[lane] * yi;
            if (lane + 32 < nb) a1 += row[lane + 32] * yi;
        }
        part[warp * NW_NB + lane] = a0;
        part[warp * NW_NB + lane + 32] = a1;
        __syncthreads();
        if (tid < NW_NB) {
            double acc = 0.0;
#pragma unroll
            for (int w = 0; w < NWARP; ++w) acc += part[w * NW_NB + tid];
            t[tid] = (tid < nb) ? y[j0 + tid] - acc : 0.0;
        }
        __syncthreads();
        const double* inv = INV + ((long long)c * npanels + pn) * NW_NB * NW_NB;
        double a = 0.0;
        if (tid < nb)
            for (int m = 0; m <= tid; ++m) a += inv[m * NW_NB + tid] * t[m];  // (U^{-T} t)_q = sum_{m <= q} inv[m][q] t_m
        __syncthreads();
        if (tid < nb) y[j0 + tid] = a;
        __syncthreads();
    }
    // backward: d_j = U_jj^{-1} (y_j - U[j-rows][right cols] d_right)
    for (int pn = np - 1; pn >= 0; --pn) {
        const int j0 = pn * NW_NB, nb = min(NW_NB, p - j0);
        for (int r = warp; r < nb; r += NWARP) {
            const double* row = Hc + (long long)(j0 + r) * ldh;
            double acc = 0.0;
            for (int m = j0 + nb + lane; m < p; m += 32) acc += row[m] * y[m];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) t[r] = y[j0 + r] - acc;
        }
        __syncthreads();
        const double* inv = INV + ((long long)c * npanels + pn) * NW_NB * NW_NB;
        double a = 0.0;
        if (tid < nb)
            for (int m = tid; m < nb; ++m) a += inv[tid * NW_NB + m] * t[m];  // upper: row q, columns m >= q
        __syncthreads();
        if (tid < nb) y[j0 + tid] = a;
        __syncthreads();
    }
    for (int j = tid; j < p; j += NW_TS) DIR[(long long)c * ldv + act[j]] = y[j];
}

// Armijo backtracking on phi(x + t d) - phi(x) (formed without cancellation), one block per column.
// q2 = d'(G_AA/n)d comes from the Newton system itself: d'Hd = -grad'd, H = G_AA/n + curvature terms.
// With l1 weights backtracking starts at min(1, t_cross) and the l1 difference t sum_j w1_j s_j d_j joins dphi;
// a step accepted at t_cross sets the coordinates that cross (nw_cross(x_j, d_j) <= t) to exactly zero.
// out[c] = {accepted (0/1), t, decrement = -grad'd, 0}.  X is updated in place when accepted.
__global__ void __launch_bounds__(NW_T) newton_linesearch_kernel(int p, int Gn, const int* __restrict__ gptr,
                                                                 double* __restrict__ X, const double* __restrict__ DIR,
                                                                 const double* __restrict__ GS, const double* __restrict__ GRAD,
                                                                 const double* __restrict__ U, const double* __restrict__ KK,
                                                                 const double* __restrict__ DP, long long ldv,
                                                                 const double* __restrict__ W2, const double* __restrict__ NRM,
                                                                 const double* __restrict__ W1, const int* __restrict__ info,
                                                                 double* __restrict__ out) {
    extern __shared__ double sh[];  // g1[Gn], g2[Gn]
    __shared__ double red[NW_T / 32];
    __shared__ double tsel;
    double* g1 = sh;
    double* g2 = sh + Gn;
    const int c = blockIdx.x, tid = threadIdx.x;
    double* x = X + (long long)c * ldv;
    const double* d = DIR + (long long)c * ldv;
    double q1 = 0.0, gd = 0.0, r1 = 0.0, r2 = 0.0, cdd = 0.0;
    const bool whole = W1 != nullptr && Gn == 1;  // Lasso's single group: the whole block walks its coordinates
    if (whole) {
        double a1 = 0.0, a2 = 0.0, ud = 0.0;
        for (int j = gptr[0] + tid; j < gptr[1]; j += NW_T) {
            const long long e = (long long)c * ldv + j;
            const double dj = d[j], xj = x[j];
            a1 += xj * dj;
            a2 += dj * dj;
            q1 += GS[e] * dj;
            gd += GRAD[e] * dj;
            const double kk = KK[e];
            if (kk >= 0.0) {
                r1 += DP[e] * xj * dj;
                r2 += DP[e] * dj * dj;
                cdd += (kk + DP[e]) * dj * dj;
                ud += U[e] * dj;
            }
        }
        a1 = nw_block_sum(a1, red);
        a2 = nw_block_sum(a2, red);
        ud = nw_block_sum(ud, red);
        if (tid == 0) {
            const double nrm = NRM[c];
            cdd -= (nrm > 0.0 ? W2[c] / nrm : 0.0) * ud * ud;  // the group's kk, as newton_prepare_kernel forms it
            g1[0] = a1;
            g2[0] = a2;
        }
    }
    for (int g = whole ? Gn : tid; g < Gn; g += NW_T) {
        const int ja = gptr[g], jb = gptr[g + 1];
        double a1 = 0.0, a2 = 0.0, ud = 0.0, kkg = 0.0;
        for (int j = ja; j < jb; ++j) {
            const long long e = (long long)c * ldv + j;
            const double dj = d[j], xj = x[j];
            a1 += xj * dj;
            a2 += dj * dj;
            q1 += GS[e] * dj;
            gd += GRAD[e] * dj;
            const double kk = KK[e];
            if (kk >= 0.0) {
                r1 += DP[e] * xj * dj;
                r2 += DP[e] * dj * dj;
                cdd += (kk + DP[e]) * dj * dj;
                ud += U[e] * dj;
                kkg = kk;
            }
        }
        cdd -= kkg * ud * ud;
        g1[g] = a1;
        g2[g] = a2;
    }
    q1 = nw_block_sum(q1, red);
    gd = nw_block_sum(gd, red);
    r1 = nw_block_sum(r1, red);
    r2 = nw_block_sum(r2, red);
    cdd = nw_block_sum(cdd, red);
    const double dec = -gd;
    const double q2 = dec - cdd;  // d'(G_AA/n)d
    const bool usable = info[c] == 0 && dec > 0.0 && isfinite(dec);
    double t = 1.0;
    double l1d = 0.0;  // sum_j w1_j s_j d_j: the l1 term's slope along d up to the first sign change
    if (W1) {
        double tc = INFINITY;
        for (int j = tid; j < p; j += NW_T) {
            const long long e = (long long)c * ldv + j;
            if (KK[e] >= 0.0) l1d += copysign(W1[e], x[j]) * d[j];
            tc = fmin(tc, nw_cross(x[j], d[j]));
        }
        l1d = nw_block_sum(l1d, red);
        tc = nw_block_min(tc, red);
        t = fmin(1.0, tc);
    }
    bool accepted = false;
    if (usable) {
        for (int ls = 0; ls < 24 && !accepted; ++ls) {
            double dpen = 0.0;
            for (int g = tid; g < Gn; g += NW_T) {
                const double nrm = NRM[(long long)c * Gn + g];
                const double dsq = 2.0 * t * g1[g] + t * t * g2[g];  // ||x_g + t d_g||^2 - ||x_g||^2
                const double nn = sqrt(fmax(nrm * nrm + dsq, 0.0));
                const double safe = nrm > 0.0 ? nrm : 1.0;
                dpen += W2[(long long)c * Gn + g] * dsq / (nn + safe);
            }
            dpen = nw_block_sum(dpen, red);
            double dphi = t * q1 + 0.5 * t * t * q2 + t * r1 + 0.5 * t * t * r2 + dpen;
            if (W1) dphi += t * l1d;
            if (dphi <= 1e-4 * t * gd)
                accepted = true;
            else
                t *= 0.5;
        }
    }
    if (tid == 0) tsel = accepted ? t : 0.0;
    __syncthreads();
    const double ts = tsel;
    if (ts > 0.0) {
        if (W1) {
            for (int j = tid; j < p; j += NW_T) x[j] = nw_cross(x[j], d[j]) <= ts ? 0.0 : x[j] + ts * d[j];
        } else {
            for (int j = tid; j < p; j += NW_T) x[j] += ts * d[j];
        }
    }
    if (tid == 0) {
        out[4 * c + 0] = accepted ? 1.0 : 0.0;
        out[4 * c + 1] = ts;
        out[4 * c + 2] = dec;
        out[4 * c + 3] = (double)info[c];
    }
}

}  // namespace slm
