// Solver-side kernels of the batched accelerated proximal-gradient method:
//   K6  prox_main_kernel + prox_momentum_kernel   (fused epilogue of one iteration)
//   K7  gap_partial_kernel + gap_final_kernel     (duality gap + convergence mask)
//       compact_* kernels: converged columns drop out of the batch (their coefficients
//       are scattered to the caller's array, active columns move to the front)
// All HBM/L2-bound.  State is feature-major [F][p][ldz] (grid columns contiguous),
// groups are contiguous feature ranges gptr[g]..gptr[g+1].
//
// Thread mapping: a block owns SC=8 adjacent grid columns (one 64-byte row
// segment) and SG=32 "group lanes"; lane gl handles whole groups, so group norms
// need no cross-thread traffic and every reduction has a fixed order
// (bit-reproducible run to run).  Per-column reductions that span blocks go
// through a small partials buffer part[f][chunk][q][ldz] and are finished by the
// consumer kernel in chunk order.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#include "../../include/sparselm_b200.h"

namespace slm {

constexpr int PROX_UR = 1;         // rows of a group in flight together in prox_main_kernel
constexpr int PROX_MINB = 4;       // resident blocks per SM prox_main_kernel is compiled for
constexpr int SC = 8;              // grid columns per block
constexpr int SG = 32;             // group lanes per block
constexpr int ST = SC * SG;        // threads per block
constexpr int kMaxChunks = 64;     // group chunks per column (partials per column)
constexpr int NQ = 9;              // partial quantities per (chunk, column): 0-4 gap pieces / restart dot of the
                                   // two-kernel iteration, 5-6 restart dots of the fused iteration (by parity),
                                   // 7-8 stationarity test of the smooth rows (gap kernels)
constexpr int MOM_ROWS = 256;      // rows per block in the momentum kernel

struct SolveDev {
    int F, p, Gn;
    int gpt;       // groups per thread in the chunked kernels
    int n_chunks;  // ceil(Gn / (SG*gpt)) <= kMaxChunks
    long long ldz, pa, g_stride;
    const double* G;
    const int* gptr;
    const double *lam1, *W1, *W2, *D2;
    double *B, *Z, *GZ, *GB, *T;  // B: working coefficients (compact column order)
    double* Bout;                 // caller's coefficient array (original column order)
    const int* colmap;            // [F][ldz] compact column -> original column (NULL: identity)
    const int* skip;              // [F][ldz] original order, columns the caller froze (may be NULL)
    double* theta[2];
    double* tmom[2];
    double* part;  // [F][n_chunks][NQ][ldz]
    double* rst;   // [F][ldz] restart dot of the last iteration, reduced over the chunks (fused iteration, after a compaction)
    int direct;    // gap kernels: GZ holds G*B itself (fused iteration), not G*Z of the momentum recurrence
    int* flag;     // 0 active, 1 converged/frozen, 3 skipped by the caller
    double *gap, *primal;
    int *n_iter, *status;
    int* counter;
    // max over the still-iterating columns of gap / (tol * scale) at a convergence check, as the
    // bit pattern of a positive double (atomicMax): lets the host pace sparse checks (may be NULL)
    unsigned long long* ratio;
    // row support of Z per block of SC columns (row-sparse Gram apply): zflag[f][j][cb] != 0
    // iff some active column of column block cb has Z[f][j][k] != 0
    unsigned char* zflag;
    int nblk;  // column blocks per row (ldz / SC)
    double tol, floor_rel;
    int K[SLM_MAX_FOLDS];
    double n_obs[SLM_MAX_FOLDS];
    double step[SLM_MAX_FOLDS];
    const double* lips_dev;  // [F] Lipschitz constants on the device (overrides step[]) or NULL
};

__device__ __forceinline__ double softt(double v, double t) {
    return v > t ? v - t : (v < -t ? v + t : 0.0);
}

// reduce over the SG group lanes for each of the SC columns; result valid for all threads
__device__ __forceinline__ double lanes_sum(double v, double (*red)[SC], int gl, int c) {
    red[gl][c] = v;
    __syncthreads();
#pragma unroll
    for (int s = SG / 2; s > 0; s >>= 1) {
        if (gl < s) red[gl][c] += red[gl + s][c];
        __syncthreads();
    }
    double r = red[0][c];
    __syncthreads();
    return r;
}
__device__ __forceinline__ double lanes_max(double v, double (*red)[SC], int gl, int c) {
    red[gl][c] = v;
    __syncthreads();
#pragma unroll
    for (int s = SG / 2; s > 0; s >>= 1) {
        if (gl < s) red[gl][c] = fmax(red[gl][c], red[gl + s][c]);
        __syncthreads();
    }
    double r = red[0][c];
    __syncthreads();
    return r;
}

// Group lanes.  GROUPED: a warp owns one group for the block's 8 columns; lane = c + 8*sub,
// the 4 sub-lanes stride over the group's rows and combine with two xor-shuffles (same
// value on every sub-lane, fixed order).  Singleton groups (Lasso): every lane is a row.
constexpr int SUB = 4;             // sub-lanes per group (GROUPED)
constexpr int GPB = SG / SUB;      // groups per block iteration (GROUPED)

// qmask names the four lanes {c, c+8, c+16, c+24} of one (group, column) quartet: the
// quartet's lanes hold identical reduced values, hence identical control flow, while
// different quartets of a warp are free to diverge (e.g. in the Newton iteration).
__device__ __forceinline__ double sub_sum(unsigned qmask, double v) {
    v += __shfl_xor_sync(qmask, v, SC);
    v += __shfl_xor_sync(qmask, v, 2 * SC);
    return v;
}
__device__ __forceinline__ double sub_max(unsigned qmask, double v) {
    v = fmax(v, __shfl_xor_sync(qmask, v, SC));
    v = fmax(v, __shfl_xor_sync(qmask, v, 2 * SC));
    return v;
}
__device__ __forceinline__ bool sub_any(unsigned qmask, bool v) {
    int x = v ? 1 : 0;
    x |= __shfl_xor_sync(qmask, x, SC);
    x |= __shfl_xor_sync(qmask, x, 2 * SC);
    return x != 0;
}

// ---- K6a: GB recurrence, gradient step, soft-threshold, group shrink, ridge -----
// writes T = beta_{k+1} and the per-chunk restart dot  sum (z - b+)(b+ - b)
template <bool GROUPED>
__global__ void __launch_bounds__(ST, PROX_MINB) prox_main_kernel(const __grid_constant__ SolveDev sp, int par) {
    const int f = blockIdx.z, chunk = blockIdx.y;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, gl = threadIdx.x / SC;
    const int k = k0 + c;
    __shared__ double red[SG][SC];
    const long long colbase = (long long)f * sp.ldz + k;
    const bool active = (k < Kf) && sp.flag[colbase] == 0;
    if (__syncthreads_and(!active)) return;

    const double theta = active ? sp.theta[par][colbase] : 0.0;
    const double inv1pt = 1.0 / (1.0 + theta);
    const double* __restrict__ cvec = sp.G + (long long)f * sp.g_stride + (long long)sp.p * sp.pa;
    const double n = sp.n_obs[f], step = sp.lips_dev ? 1.0 / sp.lips_dev[f] : sp.step[f];
    const double son = step / n;
    const long long ldz = sp.ldz;
    const int ko = (active && sp.colmap) ? sp.colmap[colbase] : k;  // original column (penalty arrays)
    // inactive lanes of a partly active block read column 0 of their fold (always valid
    // memory) so that whole warps can stay in the shuffles; they never write
    const int kk = active ? k : 0;
    const long long sbase = (long long)f * sp.p * ldz + kk;
    const long long wbase = (long long)f * sp.p * ldz + (active ? ko : 0);
    const long long gbase = (long long)f * sp.Gn * ldz + (active ? ko : 0);
    const double lam1 = (active && sp.lam1) ? sp.lam1[(long long)f * ldz + ko] : 0.0;
    const int sub = GROUPED ? (gl % SUB) : 0;
    const int gsl = GROUPED ? (gl / SUB) : gl;       // group slot of this lane
    const int gstep = GROUPED ? GPB : SG;            // groups per block iteration
    const int rstep = GROUPED ? SUB : 1;
    const unsigned qmask = 0x01010101u << c;

    constexpr int UR = GROUPED ? PROX_UR : 1;  // rows of a group whose loads are in flight together
    double dot = 0.0;
    for (int i = 0; i < sp.gpt; ++i) {
        const int g = (chunk * sp.gpt + i) * gstep + gsl;
        if (g >= sp.Gn) break;  // uniform over the sub-lanes of a group
        const int ja = sp.gptr ? sp.gptr[g] : g;
        const int jb = sp.gptr ? sp.gptr[g + 1] : g + 1;
        // rows in chunks of UR: all loads of a chunk are issued before its first store (the state
        // arrays are not restrict-qualified, a store in between would serialise the loads)
        double ss = 0.0;
        for (int j0 = ja + sub; j0 < jb; j0 += UR * rstep) {
            double gz[UR], gbo[UR], z[UR], cj[UR], w1[UR];
#pragma unroll
            for (int r = 0; r < UR; ++r) {
                const int j = j0 + r * rstep;
                if (j < jb) {
                    const long long e = sbase + (long long)j * ldz;
                    gz[r] = sp.GZ[e];
                    gbo[r] = sp.GB[e];
                    z[r] = sp.Z[e];
                    cj[r] = cvec[j];
                    w1[r] = sp.W1 ? sp.W1[wbase + (long long)j * ldz] : lam1;
                }
            }
#pragma unroll
            for (int r = 0; r < UR; ++r) {
                const int j = j0 + r * rstep;
                if (j < jb) {
                    const long long e = sbase + (long long)j * ldz;
                    const double gb = (gz[r] + theta * gbo[r]) * inv1pt;
                    const double v = z[r] - son * (gz[r] - cj[r]);
                    const double u = softt(v, step * w1[r]);
                    if (active) {
                        sp.GB[e] = gb;
                        sp.T[e] = u;  // stash; scaled below
                    }
                    ss += u * u;
                }
            }
        }
        if (GROUPED) ss = sub_sum(qmask, ss);
        const double nrm = sqrt(ss);
        const double w2 = sp.W2 ? sp.W2[gbase + (long long)g * ldz] : 0.0;
        const double d2 = sp.D2 ? sp.D2[gbase + (long long)g * ldz] : 0.0;
        double scale = nrm > 0.0 ? fmax(0.0, 1.0 - step * w2 / nrm) : 0.0;
        scale = scale / (1.0 + step * d2);
        if (active) {
            for (int j0 = ja + sub; j0 < jb; j0 += UR * rstep) {
                double t[UR], z[UR], bo[UR];
#pragma unroll
                for (int r = 0; r < UR; ++r) {
                    const int j = j0 + r * rstep;
                    if (j < jb) {
                        const long long e = sbase + (long long)j * ldz;
                        t[r] = sp.T[e];
                        z[r] = sp.Z[e];
                        bo[r] = sp.B[e];
                    }
                }
#pragma unroll
                for (int r = 0; r < UR; ++r) {
                    const int j = j0 + r * rstep;
                    if (j < jb) {
                        const double bn = scale * t[r];
                        sp.T[sbase + (long long)j * ldz] = bn;
                        dot += (z[r] - bn) * (bn - bo[r]);
                    }
                }
            }
        }
    }
    dot = lanes_sum(active ? dot : 0.0, red, gl, c);
    if (active && gl == 0)
        sp.part[(((long long)f * sp.n_chunks + chunk) * NQ + 0) * ldz + k] = dot;
}

// ---- K6b: restart test, momentum, state rotation (elementwise, coalesced) --------
// also records the row support of the new Z per column block (zflag) for the row-sparse apply
__global__ void __launch_bounds__(ST) prox_momentum_kernel(const __grid_constant__ SolveDev sp, int par) {
    const int f = blockIdx.z;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, r = threadIdx.x / SC;
    const int k = k0 + c;
    __shared__ double red[SG][SC];
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    const bool active = (k < Kf) && sp.flag[colbase] == 0;
    const int j0 = blockIdx.y * MOM_ROWS;
    const int j1 = min(j0 + MOM_ROWS, sp.p);
    if (__syncthreads_and(!active)) {
        // nothing iterates in this column block any more: its rows leave the support
        if (sp.zflag)
            for (int j = j0 + (int)threadIdx.x; j < j1; j += ST)
                sp.zflag[((long long)f * sp.p + j) * sp.nblk + blockIdx.x] = 0;
        return;
    }

    double acc = 0.0;
    if (active)
        for (int ch = r; ch < sp.n_chunks; ch += SG)
            acc += sp.part[(((long long)f * sp.n_chunks + ch) * NQ + 0) * ldz + k];
    const double dsum = lanes_sum(acc, red, r, c);
    const double tm = active ? sp.tmom[par][colbase] : 1.0;
    double tn = 0.5 * (1.0 + sqrt(1.0 + 4.0 * tm * tm));
    double th = (tm - 1.0) / tn;
    if (dsum > 0.0) {  // gradient-scheme adaptive restart (O'Donoghue & Candes)
        th = 0.0;
        tn = 1.0;
    }
    const long long sbase = (long long)f * sp.p * ldz + k;
    const unsigned lane = threadIdx.x & 31u;
#pragma unroll 1
    for (int jj = r; jj < MOM_ROWS; jj += SG) {  // uniform trip count: the ballot needs whole warps
        const int j = j0 + jj;
        const bool inb = j < j1;
        bool nz = false;
        if (inb && active) {
            const long long e = sbase + (long long)j * ldz;
            const double bn = sp.T[e];
            const double b = sp.B[e];
            const double z = bn + th * (bn - b);
            sp.Z[e] = z;
            sp.B[e] = bn;
            nz = z != 0.0;
        }
        if (sp.zflag) {
            const unsigned bal = __ballot_sync(0xffffffffu, nz);
            if (c == 0 && inb)
                sp.zflag[((long long)f * sp.p + j) * sp.nblk + blockIdx.x] =
                    (unsigned char)(((bal >> (lane & 24u)) & 0xffu) != 0u);
        }
    }
    if (active && blockIdx.y == 0 && r == 0) {
        sp.theta[par ^ 1][colbase] = th;
        sp.tmom[par ^ 1][colbase] = tn;
    }
}


// ---- K6 fused: one kernel per iteration, 40 bytes per coefficient -------------------------------
// The two-kernel iteration above materialises the extrapolated point Z = W_t + th (W_t - W_{t-1}), applies
// the Gram to it, and needs a second pass (prox_momentum) because the restart test of iteration t decides
// the momentum of Z_{t+1}.  The Gram apply is linear, so it can just as well act on the iterate itself:
//     G Z_t = (1 + th) G W_t - th G W_{t-1}.
// With W_t, W_{t-1}, G W_t, G W_{t-1} resident (two buffers each, swapped by parity), z and G z are formed on
// the fly at the START of iteration t -- when the restart test of iteration t-1 is already known -- and one
// kernel does momentum, gradient step, soft-threshold, group shrink, ridge, restart dot and the support flags
// of the new iterate: reads W_t, W_{t-1}, G W_t, G W_{t-1}, writes W_{t+1} over W_{t-1} (40 bytes per
// coefficient instead of three passes over five arrays), no T / Z round trip, one launch less.  Same
// iterates as the two-kernel form (same restart rule, same theta sequence); G W_t is exact instead of a
// recurrence, and the apply contracts over the support of W_t, a subset of that of Z_t.
struct FusedArgs {
    const double* Bcur;   // W_t
    double* Bnew;         // holds W_{t-1} on entry, W_{t+1} on exit
    const double* GBcur;  // G W_t (this iteration's apply)
    const double* GBold;  // G W_{t-1}
    double* stash;        // [F][p][ldz] scratch for groups too long for registers
    int it;               // iteration index (0: no momentum)
    int use_rst;          // restart dot of iteration it-1 from sp.rst (after a compaction) instead of the partials
};

// momentum coefficient of iteration `it` for one column: th = (t_{k-1} - 1) / t_k unless the last iteration's
// restart dot was positive.  tm = t_{k-1} (tmom of the other parity), returns th and the new t_k in tn.
__device__ __forceinline__ double fused_theta(int it, double tm, double dsum, double* tn) {
    if (it == 0) {
        *tn = tm;
        return 0.0;
    }
    double t = 0.5 * (1.0 + sqrt(1.0 + 4.0 * tm * tm));
    double th = (tm - 1.0) / t;
    if (dsum > 0.0) {  // gradient-scheme adaptive restart (O'Donoghue & Candes)
        th = 0.0;
        t = 1.0;
    }
    *tn = t;
    return th;
}

// FZ_RC: rows per lane kept in registers across the group-norm reduction (the host picks the smallest
// instantiation that covers the largest group: unused row slots still cost issue slots)
template <bool GROUPED, int FZ_RC>
__global__ void __launch_bounds__(ST, GROUPED ? (FZ_RC <= 5 ? 3 : 2) : PROX_MINB)
    prox_fused_kernel(const __grid_constant__ SolveDev sp, const __grid_constant__ FusedArgs fa, int par) {
    const int f = blockIdx.z, chunk = blockIdx.y;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, gl = threadIdx.x / SC;
    const int k = k0 + c;
    __shared__ double red[SG][SC];
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    const bool active = (k < Kf) && sp.flag[colbase] == 0;
    const int sub = GROUPED ? (gl % SUB) : (gl % 4);   // which byte of a warp ballot holds this lane's 8 columns
    const int gsl = GROUPED ? (gl / SUB) : gl;         // group slot of this lane
    const int gstep = GROUPED ? GPB : SG;              // groups per block iteration
    const int rstep = GROUPED ? SUB : 1;
    const int rsub = GROUPED ? sub : 0;
    if (__syncthreads_and(!active)) {
        // nothing iterates in this column block any more: the rows of this chunk's groups leave the support
        if (sp.zflag && c == 0)
            for (int i = 0; i < sp.gpt; ++i) {
                const int g = (chunk * sp.gpt + i) * gstep + gsl;
                if (g >= sp.Gn) break;
                const int ja = sp.gptr ? sp.gptr[g] : g, jb = sp.gptr ? sp.gptr[g + 1] : g + 1;
                for (int j = ja + rsub; j < jb; j += rstep) sp.zflag[((long long)f * sp.p + j) * sp.nblk + blockIdx.x] = 0;
            }
        return;
    }
    // restart dot of the previous iteration (every block of the column sums the same partials in the same order)
    double dsum = 0.0;
    if (fa.it > 0) {
        if (fa.use_rst) {
            dsum = active ? sp.rst[colbase] : 0.0;
        } else {
            const int slot_in = 5 + (par ^ 1);
            double acc = 0.0;
            if (active)
                for (int ch = gl; ch < sp.n_chunks; ch += SG)
                    acc += sp.part[(((long long)f * sp.n_chunks + ch) * NQ + slot_in) * ldz + k];
            dsum = lanes_sum(acc, red, gl, c);
        }
    }
    double tn;
    const double th = fused_theta(fa.it, active ? sp.tmom[par ^ 1][colbase] : 1.0, dsum, &tn);
    if (active && chunk == 0 && gl == 0) {
        sp.theta[par][colbase] = th;
        sp.tmom[par][colbase] = tn;
    }
    const double* __restrict__ cvec = sp.G + (long long)f * sp.g_stride + (long long)sp.p * sp.pa;
    const double n = sp.n_obs[f], step = sp.lips_dev ? 1.0 / sp.lips_dev[f] : sp.step[f];
    const double son = step / n;
    const int ko = (active && sp.colmap) ? sp.colmap[colbase] : k;  // original column (penalty arrays)
    const int kk = active ? k : 0;  // inactive lanes of a partly active block shadow column 0 (reads only)
    const long long sbase = (long long)f * sp.p * ldz + kk;
    const long long wbase = (long long)f * sp.p * ldz + (active ? ko : 0);
    const long long gbase = (long long)f * sp.Gn * ldz + (active ? ko : 0);
    const double lam1 = (active && sp.lam1) ? sp.lam1[(long long)f * ldz + ko] : 0.0;
    const unsigned qmask = 0x01010101u << c;
    const unsigned lane = threadIdx.x & 31u;
    const double* __restrict__ Bcur = fa.Bcur;
    const double* __restrict__ GBcur = fa.GBcur;
    const double* __restrict__ GBold = fa.GBold;

    double dot = 0.0;
    for (int i = 0; i < sp.gpt; ++i) {
        const int g = (chunk * sp.gpt + i) * gstep + gsl;
        if (GROUPED && g >= sp.Gn) break;  // uniform over the warp (a warp owns one group)
        const bool gv = g < sp.Gn;         // singleton groups: the lanes of a warp hold different rows
        const int ja = gv ? (sp.gptr ? sp.gptr[g] : g) : 0;
        const int jb = gv ? (sp.gptr ? sp.gptr[g + 1] : g + 1) : 0;
        const double w2 = (gv && sp.W2) ? sp.W2[gbase + (long long)g * ldz] : 0.0;
        const double d2 = (gv && sp.D2) ? sp.D2[gbase + (long long)g * ldz] : 0.0;
        if (!GROUPED || jb - ja <= FZ_RC * rstep) {
            // the group's rows of this lane stay in registers across the norm reduction: one pass
            constexpr int RC = GROUPED ? FZ_RC : 1;
            // four loads per row in flight for all RC rows, then the registers are recycled: bb = W_t, zz takes
            // the place of W_{t-1}, u that of G W_t
            double bb[RC], zz[RC], u[RC], gbo[RC];
            double ss = 0.0;
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                const int j = ja + rsub + r * rstep;
                bb[r] = zz[r] = u[r] = gbo[r] = 0.0;
                if (j < jb) {
                    const long long e = sbase + (long long)j * ldz;
                    bb[r] = Bcur[e];
                    zz[r] = fa.Bnew[e];
                    u[r] = GBcur[e];
                    gbo[r] = GBold[e];
                }
            }
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                const int j = ja + rsub + r * rstep;
                if (j < jb) {
                    const double w1 = sp.W1 ? sp.W1[wbase + (long long)j * ldz] : lam1;
                    const double z = bb[r] + th * (bb[r] - zz[r]);
                    const double gz = u[r] + th * (u[r] - gbo[r]);
                    const double v = z - son * (gz - cvec[j]);
                    zz[r] = z;
                    u[r] = softt(v, step * w1);
                    ss += u[r] * u[r];
                } else {
                    u[r] = 0.0;
                }
            }
            if (GROUPED) ss = sub_sum(qmask, ss);
            const double nrm = sqrt(ss);
            double scale = nrm > 0.0 ? fmax(0.0, 1.0 - step * w2 / nrm) : 0.0;
            scale = scale / (1.0 + step * d2);
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                const int j = ja + rsub + r * rstep;
                const bool inb = j < jb;
                bool nz = false;
                if (inb && active) {
                    const double bn = scale * u[r];
                    fa.Bnew[sbase + (long long)j * ldz] = bn;
                    dot += (zz[r] - bn) * (bn - bb[r]);
                    nz = bn != 0.0;
                }
                if (sp.zflag) {
                    const unsigned bal = __ballot_sync(0xffffffffu, nz);
                    if (c == 0 && inb)
                        sp.zflag[((long long)f * sp.p + j) * sp.nblk + blockIdx.x] =
                            (unsigned char)(((bal >> (lane & 24u)) & 0xffu) != 0u);
                }
            }
        } else {
            // long group (GROUPED only): u goes through the stash array, two passes
            double ss = 0.0;
            for (int j = ja + rsub; j < jb; j += rstep) {
                const long long e = sbase + (long long)j * ldz;
                const double b = Bcur[e], bo = fa.Bnew[e], gbn = GBcur[e], gbo = GBold[e];
                const double w1 = sp.W1 ? sp.W1[wbase + (long long)j * ldz] : lam1;
                const double z = b + th * (b - bo);
                const double gz = gbn + th * (gbn - gbo);
                const double u = softt(z - son * (gz - cvec[j]), step * w1);
                if (active) fa.stash[e] = u;
                ss += u * u;
            }
            ss = sub_sum(qmask, ss);
            const double nrm = sqrt(ss);
            double scale = nrm > 0.0 ? fmax(0.0, 1.0 - step * w2 / nrm) : 0.0;
            scale = scale / (1.0 + step * d2);
            const int trips = (jb - ja + rstep - 1) / rstep;  // uniform over the warp: the ballot needs whole warps
            for (int t = 0; t < trips; ++t) {
                const int j = ja + rsub + t * rstep;
                const bool inb = j < jb;
                bool nz = false;
                if (inb && active) {
                    const long long e = sbase + (long long)j * ldz;
                    const double b = Bcur[e], bo = fa.Bnew[e];
                    const double bn = scale * fa.stash[e];
                    const double z = b + th * (b - bo);
                    fa.Bnew[e] = bn;
                    dot += (z - bn) * (bn - b);
                    nz = bn != 0.0;
                }
                if (sp.zflag) {
                    const unsigned bal = __ballot_sync(0xffffffffu, nz);
                    if (c == 0 && inb)
                        sp.zflag[((long long)f * sp.p + j) * sp.nblk + blockIdx.x] =
                            (unsigned char)(((bal >> (lane & 24u)) & 0xffu) != 0u);
                }
            }
        }
    }
    dot = lanes_sum(active ? dot : 0.0, red, gl, c);
    if (active && gl == 0)
        sp.part[(((long long)f * sp.n_chunks + chunk) * NQ + 5 + par) * ldz + k] = dot;
}

// columns flagged at this convergence check: their final iterate goes into BOTH iterate buffers, so that
// whichever buffer is "current" when they are collected (compaction, end of the solve) holds it
__global__ void __launch_bounds__(ST) settle_done_kernel(const __grid_constant__ SolveDev sp, const double* __restrict__ src,
                                                         double* __restrict__ dst) {
    const int f = blockIdx.z;
    const int Kf = sp.K[f];
    const int k = blockIdx.x * SC + threadIdx.x % SC;
    const int r = threadIdx.x / SC;
    if (k >= Kf || sp.flag[(long long)f * sp.ldz + k] != 1) return;
    const long long sb = (long long)f * sp.p * sp.ldz + k;
    const int j0 = blockIdx.y * MOM_ROWS, j1 = min(j0 + MOM_ROWS, sp.p);
    for (int j = j0 + r; j < j1; j += SG) dst[sb + (long long)j * sp.ldz] = src[sb + (long long)j * sp.ldz];
}

// restart dot of iteration `par` summed over the chunks into sp.rst (before a compaction renumbers the columns)
__global__ void restart_reduce_kernel(const __grid_constant__ SolveDev sp, int par) {
    const int f = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= sp.K[f]) return;
    double acc = 0.0;
    for (int ch = 0; ch < sp.n_chunks; ++ch) acc += sp.part[(((long long)f * sp.n_chunks + ch) * NQ + 5 + par) * sp.ldz + k];
    sp.rst[(long long)f * sp.ldz + k] = acc;
}

// fused -> two-kernel state at the start of iteration `it` (the cluster / cooperative kernels and the
// two-kernel iteration work on Z, B, GB, theta): Z = W_t + th (W_t - W_{t-1}), B = W_t, GB = G W_{t-1},
// theta[par] = th, tmom[par] = t_k.  Bcur / Bold / GBold may alias sp.B / sp.GB (element-wise, read before write).
__global__ void __launch_bounds__(ST) fused_to_classic_kernel(const __grid_constant__ SolveDev sp, const double* Bcur,
                                                              const double* Bold, const double* GBold, int it,
                                                              int par, int use_rst) {
    const int f = blockIdx.z;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, r = threadIdx.x / SC;
    const int k = k0 + c;
    __shared__ double red[SG][SC];
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    const bool active = (k < Kf) && sp.flag[colbase] == 0;
    double dsum = 0.0;
    if (it > 0) {
        if (use_rst) {
            dsum = active ? sp.rst[colbase] : 0.0;
        } else {
            double acc = 0.0;
            if (active)
                for (int ch = r; ch < sp.n_chunks; ch += SG)
                    acc += sp.part[(((long long)f * sp.n_chunks + ch) * NQ + 5 + (par ^ 1)) * ldz + k];
            dsum = lanes_sum(acc, red, r, c);
        }
    }
    double tn;
    const double th = fused_theta(it, active ? sp.tmom[par ^ 1][colbase] : 1.0, dsum, &tn);
    const long long sb = (long long)f * sp.p * ldz + k;
    const int j0 = blockIdx.y * MOM_ROWS, j1 = min(j0 + MOM_ROWS, sp.p);
    if (k < Kf && sp.flag[colbase] != 3)  // columns the caller froze never entered the iterate buffers
        for (int j = j0 + r; j < j1; j += SG) {
            const long long e = sb + (long long)j * ldz;
            const double b = Bcur[e], bo = Bold[e], gbo = GBold[e];
            sp.Z[e] = active ? b + th * (b - bo) : b;
            sp.B[e] = b;
            sp.GB[e] = gbo;
        }
    if (active && blockIdx.y == 0 && r == 0) {
        sp.theta[par][colbase] = th;
        sp.tmom[par][colbase] = tn;
    }
}

// ---- row support of Z for the row-sparse Gram apply -----------------------------------
// flags from scratch (start of a solve, after a compaction, final certificate): every
// column k < K[f] counts
__global__ void __launch_bounds__(256) zflags_kernel(const __grid_constant__ SolveDev sp,
                                                     const double* __restrict__ Zsrc) {
    const int f = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)sp.p * sp.nblk) return;
    const int j = (int)(i / sp.nblk), cb = (int)(i - (long long)j * sp.nblk);
    const int Kf = sp.K[f];
    bool nz = false;
    const double* row = Zsrc + ((long long)f * sp.p + j) * sp.ldz;
    for (int k = cb * SC; k < min(cb * SC + SC, Kf); ++k) nz |= row[k] != 0.0;
    sp.zflag[((long long)f * sp.p + j) * sp.nblk + cb] = nz ? 1 : 0;
}

// ordered list of the support rows of every (fold, column chunk): chunk cc covers the column
// blocks [cc*wb, (cc+1)*wb); sidx[(f*ncc + cc)*p + i] ascending, scount[f*ncc + cc] entries.
// stat accumulates sum(rows x real columns) = executed contraction length (for the roofline).
__global__ void __launch_bounds__(1024) support_list_kernel(const __grid_constant__ SolveDev sp, int wb, int ncc,
                                                            int* __restrict__ sidx, int* __restrict__ scount,
                                                            unsigned long long* __restrict__ stat) {
    const int f = blockIdx.y, cc = blockIdx.x;
    const int Kf = sp.K[f];
    const int nb_f = (Kf + SC - 1) / SC;
    const int b0 = cc * wb, b1 = min(b0 + wb, nb_f);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* out = sidx + ((long long)f * ncc + cc) * sp.p;
    if (b0 >= nb_f) {
        if (tid == 0) scount[f * ncc + cc] = 0;
        return;
    }
    __shared__ int wtot[32];
    __shared__ int woff[32];
    __shared__ int base_s, btot;
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int j0 = 0; j0 < sp.p; j0 += 1024) {
        const int j = j0 + tid;
        bool nz = false;
        if (j < sp.p) {
            const unsigned char* fl = sp.zflag + ((long long)f * sp.p + j) * sp.nblk;
            for (int b = b0; b < b1; ++b) nz |= fl[b] != 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, nz);
        if (lane == 0) wtot[warp] = __popc(bal);
        __syncthreads();
        if (warp == 0) {
            int v = wtot[lane], x = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            woff[lane] = x - v;
            if (lane == 31) btot = x;
        }
        __syncthreads();
        const int base = base_s;
        if (nz) out[base + woff[warp] + __popc(bal & ((1u << lane) - 1u))] = j;
        __syncthreads();
        if (tid == 0) base_s = base + btot;
        __syncthreads();
    }
    if (tid == 0) {
        scount[f * ncc + cc] = base_s;
        if (stat) atomicAdd(stat, (unsigned long long)base_s * (unsigned long long)(min(b1 * SC, Kf) - b0 * SC));
    }
}

// dual norm of one group: smallest nu with || S(|g|, nu*w1) ||_2 <= nu*w2, by a
// monotone Newton iteration from a lower bound (psi is convex and decreasing),
// finished on the feasible side.  gfun(j) returns |g_j|, wfun(j) returns w1_j; rows
// ja+sub, ja+sub+rstep, ... belong to this lane and partial sums are combined over the
// sub-lanes, so all sub-lanes of a group take identical decisions.
template <bool GROUPED, typename GF, typename WF>
__device__ __forceinline__ double group_dual_newton(unsigned qmask, int ja, int jb, int sub, int rstep, double w2,
                                                    double lo, double hi, GF gfun, WF wfun) {
    double nu = lo;
    for (int it = 0; it < 50; ++it) {
        double s2 = 0.0, sw = 0.0;
        for (int j = ja + sub; j < jb; j += rstep) {
            const double w = wfun(j);
            const double u = gfun(j) - nu * w;
            if (u > 0.0) {
                s2 += u * u;
                sw += w * u;
            }
        }
        if (GROUPED) {
            s2 = sub_sum(qmask, s2);
            sw = sub_sum(qmask, sw);
        }
        const double s = sqrt(s2);
        const double psi = s - nu * w2;
        if (!(psi > 0.0)) break;
        const double dpsi = -sw / s - w2;
        const double nn = nu - psi / dpsi;
        if (!(nn > nu)) break;
        nu = nn;
    }
    // finish on the feasible side
    double bump = 4e-16;
    for (int t = 0; t < 12; ++t) {
        const double cand = nu * (1.0 + bump);
        double s2 = 0.0;
        for (int j = ja + sub; j < jb; j += rstep) {
            const double u = gfun(j) - cand * wfun(j);
            if (u > 0.0) s2 += u * u;
        }
        if (GROUPED) s2 = sub_sum(qmask, s2);
        if (sqrt(s2) <= cand * w2) return fmin(cand, hi);
        bump *= 8.0;
    }
    return hi;
}

// Smooth rows: w1_j = 0 in a group with w2_g = 0 (a group left unpenalised, or an unpenalised coordinate of a
// pure-l1 group; the ridge D2 may be anything).  Their dual constraint is g_j = 0, which a scaled residual meets
// only to rounding: taken into omega, such a row makes the dual norm +inf (dual 0, gap = primal) at the optimum.
// So they stay out of omega, and a column is converged only if in addition every smooth row is stationary to
// the rounding bound of (c - G b)_j (Cauchy-Schwarz: |G_jk| <= sqrt(G_jj G_kk)):
//     |g_j| <= tau_j = kSmoothKappa * eps * (|c_j| + sqrt(G_jj) * S) / n,   S = sum_k sqrt(G_kk) |b_k|.
// gap_partial_kernel keeps per chunk its share of S (slot 7) and the largest S a smooth row needs to pass,
// (n |g_j| / (kSmoothKappa eps) - |c_j|) / sqrt(G_jj) (slot 8); gap_final_kernel compares the two.  The bound is
// loose: converged fits leave |g_j| at most 0.19 tau_j(kappa = 1) (B200, test_zero_weight_group_fits_converge;
// 0.02-0.08 in the float64 model), so kappa = 64 leaves room for the GB recurrence of the small-design and
// two-kernel checks and still asks for stationarity to within ~1e-14 relative.
constexpr double kSmoothKappa = 64.0;
constexpr double kSmoothTau = kSmoothKappa * 2.220446049250313e-16;  // kappa * eps

// ---- K7a: per-chunk pieces of the duality gap of B_k ------------------------------
// G B_k comes from the momentum recurrence (GZ, GB_{k-1}, theta) or, in final mode
// (Z == B), from GZ directly.
template <bool GROUPED>
__global__ void __launch_bounds__(ST) gap_partial_kernel(const __grid_constant__ SolveDev sp, int par,
                                                         int final_mode) {
    const int f = blockIdx.z, chunk = blockIdx.y;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, gl = threadIdx.x / SC;
    const int k = k0 + c;
    __shared__ double red[SG][SC];
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    // loop mode: compact columns still iterating; final mode: every original column the
    // caller did not freeze (state arrays are then in original order, colmap == NULL)
    bool active = k < Kf;
    if (active) active = final_mode ? !(sp.skip && sp.skip[colbase]) : (sp.flag[colbase] == 0);
    if (__syncthreads_and(!active)) return;

    const double theta = (active && !final_mode) ? sp.theta[par][colbase] : 0.0;
    const double inv1pt = 1.0 / (1.0 + theta);
    const double* __restrict__ cvec = sp.G + (long long)f * sp.g_stride + (long long)sp.p * sp.pa;
    const double n = sp.n_obs[f];
    const double inv_n = 1.0 / n;
    const int ko = (active && sp.colmap) ? sp.colmap[colbase] : k;
    const int kk = active ? k : 0;  // inactive lanes shadow column 0 (reads only)
    const long long sbase = (long long)f * sp.p * ldz + kk;
    const long long wbase = (long long)f * sp.p * ldz + (active ? ko : 0);
    const long long gbase = (long long)f * sp.Gn * ldz + (active ? ko : 0);
    const double lam1 = (active && sp.lam1) ? sp.lam1[(long long)f * ldz + ko] : 0.0;
    const int sub = GROUPED ? (gl % SUB) : 0;
    const int gsl = GROUPED ? (gl / SUB) : gl;
    const int gstep = GROUPED ? GPB : SG;
    const int rstep = GROUPED ? SUB : 1;
    const unsigned qmask = 0x01010101u << c;

    auto gb_at = [&](long long e) {
        const double gz = sp.GZ[e];
        return (final_mode || sp.direct) ? gz : (gz + theta * sp.GB[e]) * inv1pt;
    };

    double cb = 0.0, bgb = 0.0, pen = 0.0, ridge = 0.0, lbmax = 0.0;
    for (int i = 0; i < sp.gpt; ++i) {
        const int g = (chunk * sp.gpt + i) * gstep + gsl;
        if (g >= sp.Gn) break;
        const int ja = sp.gptr ? sp.gptr[g] : g;
        const int jb = sp.gptr ? sp.gptr[g + 1] : g + 1;
        const double w2 = sp.W2 ? sp.W2[gbase + (long long)g * ldz] : 0.0;
        const double d2 = sp.D2 ? sp.D2[gbase + (long long)g * ldz] : 0.0;
        double ss = 0.0, gg2 = 0.0, ratio = 0.0, ww2 = 0.0;
        bool anyinf = false;
        for (int j = ja + sub; j < jb; j += rstep) {
            const long long e = sbase + (long long)j * ldz;
            const double gb = gb_at(e);
            const double b = sp.B[e];
            const double cj = cvec[j];
            const double w1 = sp.W1 ? sp.W1[wbase + (long long)j * ldz] : lam1;
            cb += cj * b;
            bgb += b * gb;
            pen += w1 * fabs(b);
            ss += b * b;
            const double gj = fabs((cj - gb) * inv_n - d2 * b);
            gg2 += gj * gj;
            ww2 += w1 * w1;
            if (gj > 0.0) {
                if (w1 > 0.0)
                    ratio = fmax(ratio, gj / w1);
                else if (w2 > 0.0)  // w2 = 0: a smooth row, tested below
                    anyinf = true;
            }
        }
        if (GROUPED) {
            ss = sub_sum(qmask, ss);
            gg2 = sub_sum(qmask, gg2);
            ww2 = sub_sum(qmask, ww2);
            ratio = sub_max(qmask, ratio);
            anyinf = sub_any(qmask, anyinf);
        }
        if (sub == 0) {  // per-group terms are counted once
            pen += w2 * sqrt(ss);
            ridge += d2 * ss;
        }
        // lower bound of this group's dual norm (exact when a closed form exists)
        double lb;
        const double gn = sqrt(gg2);
        if (gg2 == 0.0)
            lb = 0.0;
        else if (w2 <= 0.0)
            lb = anyinf ? INFINITY : ratio;
        else if (ww2 == 0.0)
            lb = gn / w2;
        else
            lb = gn / (w2 + sqrt(ww2));
        lbmax = fmax(lbmax, lb);
    }
    cb = lanes_sum(active ? cb : 0.0, red, gl, c);
    bgb = lanes_sum(active ? bgb : 0.0, red, gl, c);
    pen = lanes_sum(active ? pen : 0.0, red, gl, c);
    ridge = lanes_sum(active ? ridge : 0.0, red, gl, c);
    double* dst = sp.part + (((long long)f * sp.n_chunks + chunk) * NQ) * ldz + k;
    if (active && gl == 0) {
        dst[0 * ldz] = cb;
        dst[1 * ldz] = bgb;
        dst[2 * ldz] = pen;
        dst[3 * ldz] = ridge;
    }
    if (!active) lbmax = 0.0;
    // block-wide threshold: only groups whose upper bound exceeds it can hold the max
    const double thr = lanes_max(lbmax, red, gl, c);
    double omega = lbmax;
    // second pass: Newton refinement of the groups that can hold the max, the smooth-row test
    const double* __restrict__ gdiag = sp.G + (long long)f * sp.g_stride;  // G_jj at gdiag[j * (pa + 1)]
    double sroot = 0.0, sneed = 0.0;
    for (int i = 0; i < sp.gpt; ++i) {
        const int g = (chunk * sp.gpt + i) * gstep + gsl;
        if (g >= sp.Gn) break;
        const double w2 = sp.W2 ? sp.W2[gbase + (long long)g * ldz] : 0.0;
        const int ja = sp.gptr ? sp.gptr[g] : g;
        const int jb = sp.gptr ? sp.gptr[g + 1] : g + 1;
        const double d2 = sp.D2 ? sp.D2[gbase + (long long)g * ldz] : 0.0;
        auto gfun = [&](int j) {
            const long long e = sbase + (long long)j * ldz;
            return fabs((cvec[j] - gb_at(e)) * inv_n - d2 * sp.B[e]);
        };
        auto wfun = [&](int j) { return sp.W1 ? sp.W1[wbase + (long long)j * ldz] : lam1; };
        double gg2 = 0.0, ratio = 0.0, ww2 = 0.0;
        bool anyinf = false;
        for (int j = ja + sub; j < jb; j += rstep) {
            const double gj = gfun(j), w1 = wfun(j);
            const double dj = sqrt(gdiag[(long long)j * (sp.pa + 1)]);
            sroot += dj * fabs(sp.B[sbase + (long long)j * ldz]);
            gg2 += gj * gj;
            ww2 += w1 * w1;
            if (gj > 0.0) {
                if (w1 > 0.0) {
                    ratio = fmax(ratio, gj / w1);
                } else {
                    anyinf = true;
                    if (w2 <= 0.0)  // smooth row (fmax drops the NaN of 0 / 0 for an all-zero column)
                        sneed = fmax(sneed, (gj / (inv_n * kSmoothTau) - fabs(cvec[j])) / dj);
                }
            }
        }
        if (GROUPED) {
            gg2 = sub_sum(qmask, gg2);
            ww2 = sub_sum(qmask, ww2);
            ratio = sub_max(qmask, ratio);
            anyinf = sub_any(qmask, anyinf);
        }
        const double gn = sqrt(gg2);
        double hi = w2 > 0.0 ? gn / w2 : 0.0;
        if (!anyinf && ratio < hi) hi = ratio;
        // identical on the four sub-lanes of the quartet (all inputs are quartet-reduced)
        const bool refine = active && w2 > 0.0 && gg2 > 0.0 && ww2 > 0.0 && hi > thr;
        if (refine) {
            const double lo = gn / (w2 + sqrt(ww2));
            omega = fmax(omega, group_dual_newton<GROUPED>(qmask, ja, jb, sub, rstep, w2, lo, hi, gfun, wfun));
        }
    }
    omega = lanes_max(active ? omega : 0.0, red, gl, c);
    sroot = lanes_sum(active ? sroot : 0.0, red, gl, c);
    sneed = lanes_max(active ? sneed : 0.0, red, gl, c);
    if (active && gl == 0) {
        dst[4 * ldz] = omega;
        dst[7 * ldz] = sroot;
        dst[8 * ldz] = sneed;
    }
}

// ---- K7b: finish the gap per column, set convergence flags --------------------------
// counter[f] receives the number of columns of fold f that are still iterating.
__global__ void gap_final_kernel(const __grid_constant__ SolveDev sp, int it, int final_mode) {
    const int f = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= sp.K[f]) return;
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    const bool active = final_mode ? !(sp.skip && sp.skip[colbase]) : (sp.flag[colbase] == 0);
    if (!active) return;
    const int ko = sp.colmap ? sp.colmap[colbase] : k;
    const long long obase = (long long)f * ldz + ko;
    double cb = 0.0, bgb = 0.0, pen = 0.0, ridge = 0.0, omega = 0.0, sroot = 0.0, sneed = 0.0;
    for (int ch = 0; ch < sp.n_chunks; ++ch) {
        const double* src = sp.part + (((long long)f * sp.n_chunks + ch) * NQ) * ldz + k;
        cb += src[0 * ldz];
        bgb += src[1 * ldz];
        pen += src[2 * ldz];
        ridge += src[3 * ldz];
        omega = fmax(omega, src[4 * ldz]);
        sroot += src[7 * ldz];
        sneed = fmax(sneed, src[8 * ldz]);
    }
    const bool smooth_ok = sneed <= sroot;  // every smooth row stationary to rounding (none: 0 <= S)
    const double* Gf = sp.G + (long long)f * sp.g_stride;
    const double n = sp.n_obs[f];
    const double yty = Gf[(long long)sp.p * sp.pa + sp.p];
    const double rr = yty - 2.0 * cb + bgb;
    const double rr_aug = rr + n * ridge;
    const double yr = yty - cb;
    const double P = rr_aug / (2.0 * n) + pen;
    double s = omega > 1.0 ? 1.0 / omega : 1.0;
    if (!(omega < INFINITY)) s = 0.0;
    const double D = (2.0 * s * yr - s * s * rr_aug) / (2.0 * n);
    const double gap = P - D;
    // P and D are evaluated from Gram quantities: yty - 2 c'b + b'Gb carries a rounding error of
    // a few eps * yty, so no gap below that can be certified.  The scale of the relative test
    // never goes under (4e-15 / tol) * yty/2n, i.e. tol * scale >= 4e-15 * yty/2n (18 eps: the
    // Gram entries themselves are n-term sums; measured on the README grid, where gaps of
    // noise-free data with a vanishing penalty stall between 1e-15 and 4e-15 yty/2n).
    const double scale = fmax(fabs(P), fmax(sp.floor_rel, 4e-15 / sp.tol) * yty / (2.0 * n));
    const bool finite = isfinite(P) && isfinite(gap);
    const bool conv = finite && gap <= sp.tol * scale && smooth_ok;
    if (sp.gap) sp.gap[obase] = gap;
    if (sp.primal) sp.primal[obase] = P;
    if (!final_mode) {
        if (conv || !finite) {
            sp.flag[colbase] = 1;
            if (sp.n_iter) sp.n_iter[obase] = it;
            if (sp.status) sp.status[obase] = finite ? 0 : 2;
        } else {
            atomicAdd(sp.counter + f, 1);
            if (sp.ratio) atomicMax(sp.ratio, (unsigned long long)__double_as_longlong(gap / (sp.tol * scale)));
        }
    } else {
        const bool undecided = sp.status ? sp.status[obase] == -1 : true;
        if (undecided && sp.n_iter) sp.n_iter[obase] = it;  // not flagged inside the loop
        // the exact certificate has the last word.  A column the loop flagged at `tol` from the
        // momentum recurrence of G*B keeps its status while the exact product agrees within 4 tol
        // (the two differ by the rounding of the recurrence); beyond that the recurrence has
        // drifted and the column is reported as not converged.  Columns the loop never flagged
        // are judged at tol.
        const bool ok = undecided ? conv : (finite && gap <= 4.0 * sp.tol * scale && smooth_ok);
        if (sp.status && (undecided || !ok)) sp.status[obase] = !finite ? 2 : (ok ? 0 : 1);
        if (!ok) atomicAdd(sp.counter + f, 1);
    }
}

// ---- compaction ------------------------------------------------------------------------
// src[f][kc] = current index of the kc-th still-active column of fold f (kc < newK[f]).
__global__ void compact_plan_kernel(const __grid_constant__ SolveDev sp, int* __restrict__ src,
                                    int* __restrict__ newK) {
    const int f = blockIdx.x;
    if (threadIdx.x != 0) return;
    const long long base = (long long)f * sp.ldz;
    int kc = 0;
    for (int k = 0; k < sp.K[f]; ++k)
        if (sp.flag[base + k] == 0) src[base + kc++] = k;
    newK[f] = kc;
}

// copy finished columns of the working B to the caller's array (original positions).
// all != 0: every column that is not caller-frozen (end of the solve).
__global__ void __launch_bounds__(ST) scatter_done_kernel(const __grid_constant__ SolveDev sp, int all) {
    const int f = blockIdx.z;
    const int Kf = sp.K[f];
    const int k0 = blockIdx.x * SC;
    if (k0 >= Kf) return;
    const int c = threadIdx.x % SC, r = threadIdx.x / SC;
    const int k = k0 + c;
    if (k >= Kf) return;
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    const int flag = sp.flag[colbase];
    if (flag == 3 || (!all && flag == 0)) return;
    const int ko = sp.colmap ? sp.colmap[colbase] : k;
    const long long sb = (long long)f * sp.p * ldz + k, ob = (long long)f * sp.p * ldz + ko;
    const int j0 = blockIdx.y * MOM_ROWS;
    const int j1 = min(j0 + MOM_ROWS, sp.p);
    for (int j = j0 + r; j < j1; j += SG) sp.Bout[ob + (long long)j * ldz] = sp.B[sb + (long long)j * ldz];
}

// in-place left shift of the active columns of one state array row (src is increasing)
__global__ void compact_move_kernel(const __grid_constant__ SolveDev sp, const int* __restrict__ src,
                                    const int* __restrict__ newK) {
    const int f = blockIdx.z, a = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= sp.p) return;
    const int nk = newK[f];
    if (nk == sp.K[f]) return;
    double* arr = a == 0 ? sp.Z : (a == 1 ? sp.B : sp.GB);
    double* row = arr + ((long long)f * sp.p + j) * sp.ldz;
    const int* sf = src + (long long)f * sp.ldz;
    for (int kc = 0; kc < nk; ++kc) row[kc] = row[sf[kc]];
}

__global__ void compact_cols_kernel(const __grid_constant__ SolveDev sp, const int* __restrict__ src,
                                    const int* __restrict__ newK, int* __restrict__ colmap) {
    const int f = blockIdx.x;
    if (threadIdx.x != 0) return;
    const int nk = newK[f];
    if (nk == sp.K[f]) return;
    const long long base = (long long)f * sp.ldz;
    for (int kc = 0; kc < nk; ++kc) {
        const int k = src[base + kc];
        for (int par = 0; par < 2; ++par) {
            sp.theta[par][base + kc] = sp.theta[par][base + k];
            sp.tmom[par][base + kc] = sp.tmom[par][base + k];
        }
        if (sp.rst) sp.rst[base + kc] = sp.rst[base + k];
        colmap[base + kc] = colmap[base + k];
        sp.flag[base + kc] = 0;
    }
}

// ---- small designs: many iterations per launch ---------------------------------------
// For p <= kSmallPMax one CTA owns one (fold, grid column) problem and keeps the whole Gram
// in shared memory: it runs n_inner complete iterations (Gram apply, GB recurrence, gradient
// step, soft-threshold, group shrink, ridge, restart test, momentum) without leaving the SM.
// The arithmetic is that of gemm apply + prox_main_kernel + prox_momentum_kernel; only the
// parallel decomposition differs (threads over features, the contraction split over
// `nsplit` thread groups).  State on entry/exit = the state at the top of an iteration with
// parity `par` / `par ^ (n_inner & 1)`, so the regular kernels (convergence check every so
// many iterations) interleave freely.  Ill-conditioned small problems need 1e4-1e5
// iterations: at ~0.3 us per fused iteration that is tens of ms instead of seconds of
// launch latency.
constexpr int kSmallPMax = 160;

__host__ __device__ inline size_t fista_small_smem(int p, int p32, int nsplit) {
    return sizeof(double) * ((size_t)p * p32 + (size_t)p32 * (2 + nsplit) + 64);
}

template <bool GROUPED>
__global__ void __launch_bounds__(256) fista_small_kernel(const __grid_constant__ SolveDev sp, int par, int n_inner,
                                                          int p32, int nsplit) {
    extern __shared__ __align__(16) double sm[];
    const int f = blockIdx.y, k = blockIdx.x;
    if (k >= sp.K[f]) return;
    const long long ldz = sp.ldz;
    const long long colbase = (long long)f * ldz + k;
    if (sp.flag[colbase] != 0) return;
    const int p = sp.p;
    double* Gs = sm;                          // [p][p32]: Gs[j][i] = G[j][i] (symmetric)
    double* zs = Gs + (size_t)p * p32;        // [p32] current z
    double* us = zs + p32;                    // [p32] soft-thresholded gradient step
    double* parts = us + p32;                 // [nsplit][p32] partial contractions
    double* red = parts + (size_t)nsplit * p32;  // [64] reductions / broadcast
    const int tid = threadIdx.x, nt = blockDim.x;
    const int row = tid % p32, split = tid / p32;
    const bool valid = row < p && split < nsplit;
    const bool owner = valid && split == 0;
    const double* __restrict__ Gf = sp.G + (long long)f * sp.g_stride;
    for (int e = tid; e < p * p; e += nt) {
        const int j = e / p, i = e - j * p;
        Gs[(size_t)j * p32 + i] = Gf[(long long)j * sp.pa + i];
    }
    const int ko = sp.colmap ? sp.colmap[colbase] : k;
    const double n = sp.n_obs[f], step = sp.lips_dev ? 1.0 / sp.lips_dev[f] : sp.step[f];
    const double son = step / n;
    const long long sbase = (long long)f * p * ldz + k;
    double zi = 0.0, bi = 0.0, gbi = 0.0, cj = 0.0, tw1 = 0.0, tw2 = 0.0, rd = 1.0;
    int ja = row, jb = row + 1;
    if (owner) {
        const long long e = sbase + (long long)row * ldz;
        zi = sp.Z[e];
        bi = sp.B[e];
        gbi = sp.GB[e];
        cj = Gf[(long long)p * sp.pa + row];
        const double w1 = sp.W1 ? sp.W1[(long long)f * p * ldz + (long long)row * ldz + ko]
                                : (sp.lam1 ? sp.lam1[(long long)f * ldz + ko] : 0.0);
        tw1 = step * w1;
        int g = row;
        if (GROUPED) {
            int lo = 0, hi = sp.Gn - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (sp.gptr[mid] <= row)
                    lo = mid;
                else
                    hi = mid - 1;
            }
            g = lo;
            ja = sp.gptr[g];
            jb = sp.gptr[g + 1];
        }
        const long long gbase = (long long)f * sp.Gn * ldz + (long long)g * ldz + ko;
        tw2 = step * (sp.W2 ? sp.W2[gbase] : 0.0);
        rd = 1.0 / (1.0 + step * (sp.D2 ? sp.D2[gbase] : 0.0));
    }
    if (tid < p32) zs[tid] = owner ? zi : 0.0;
    if (tid == 0) {
        red[32] = sp.theta[par][colbase];
        red[33] = sp.tmom[par][colbase];
    }
    __syncthreads();
    double theta = red[32], tm = red[33];
    const int warp = tid >> 5, lane = tid & 31, nwarp = (nt + 31) >> 5;

#pragma unroll 1
    for (int it = 0; it < n_inner; ++it) {
        // Gram apply: gz_row = sum_j G[j][row] z_j, the contraction split over nsplit thread groups
        double a0 = 0.0, a1 = 0.0;
        if (valid) {
            int j = split;
            for (; j + nsplit < p; j += 2 * nsplit) {
                a0 += Gs[(size_t)j * p32 + row] * zs[j];
                a1 += Gs[(size_t)(j + nsplit) * p32 + row] * zs[j + nsplit];
            }
            if (j < p) a0 += Gs[(size_t)j * p32 + row] * zs[j];
        }
        double gz = a0 + a1;
        if (nsplit > 1) {
            if (valid) parts[(size_t)split * p32 + row] = gz;
            __syncthreads();
            if (owner) {
                gz = parts[row];
                for (int s2 = 1; s2 < nsplit; ++s2) gz += parts[(size_t)s2 * p32 + row];
            }
        }
        double u = 0.0;
        if (owner) {
            gbi = (gz + theta * gbi) / (1.0 + theta);
            u = softt(zi - son * (gz - cj), tw1);
            us[row] = u;
        }
        __syncthreads();
        double bn = 0.0, d = 0.0;
        if (owner) {
            double ss = 0.0;
            if (GROUPED) {
                for (int j = ja; j < jb; ++j) ss += us[j] * us[j];
            } else {
                ss = u * u;
            }
            const double nrm = sqrt(ss);
            const double scale = (nrm > 0.0 ? fmax(0.0, 1.0 - tw2 / nrm) : 0.0) * rd;
            bn = scale * u;
            d = (zi - bn) * (bn - bi);
        }
        // restart test: block sum of d in a fixed order
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        if (lane == 0) red[warp] = d;
        __syncthreads();
        if (tid == 0) {
            double dsum = 0.0;
            for (int w = 0; w < nwarp; ++w) dsum += red[w];
            double tn = 0.5 * (1.0 + sqrt(1.0 + 4.0 * tm * tm));
            double th = (tm - 1.0) / tn;
            if (dsum > 0.0) {  // gradient-scheme adaptive restart
                th = 0.0;
                tn = 1.0;
            }
            red[32] = th;
            red[33] = tn;
        }
        __syncthreads();
        theta = red[32];
        tm = red[33];
        if (owner) {
            zi = bn + theta * (bn - bi);
            bi = bn;
            zs[row] = zi;
        }
        __syncthreads();
    }
    if (owner) {
        const long long e = sbase + (long long)row * ldz;
        sp.Z[e] = zi;
        sp.B[e] = bi;
        sp.GB[e] = gbi;
    }
    if (tid == 0) {
        const int po = par ^ (n_inner & 1);
        sp.theta[po][colbase] = theta;
        sp.tmom[po][colbase] = tm;
    }
}

}  // namespace slm
