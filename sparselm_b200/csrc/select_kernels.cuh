// Stability selection: selection counts of the coefficient tables of one chunk of subsample fits
// (slm_support_counts, DESIGN section 2 item 17).
//
// coef is [F][p][ldz] as the solve returns it (fit f, feature j, candidate column k).  Coefficient j of
// fit (f, k) is selected iff |coef| > rel_tol * max_j' |coef[f][j'][k]|; an all-zero fit selects nothing
// and a NaN coefficient is never selected.  Columns k >= K (batch padding) are never read.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace slm {

constexpr int SEL_ROWS = 8;    // warps (rows) of a block of both kernels
constexpr int SEL_RPT = 16;    // rows each thread of the max kernel walks

// Stage 1: colmax[f][k] = max_j |coef[f][j][k]| (NaN ignored), for k < K.  A warp reads 32 adjacent columns of a
// row; a block reduces SEL_ROWS * SEL_RPT rows and merges into colmax (zeroed by the caller) with an integer
// atomicMax on the bit pattern: non-negative doubles order like their bits, and a max is exact, so the result does
// not depend on the order of the merges.
__global__ void __launch_bounds__(32 * SEL_ROWS) support_colmax_kernel(const double* __restrict__ coef, int64_t p,
                                                                       int64_t ldz, int K,
                                                                       unsigned long long* __restrict__ colmax) {
    __shared__ double part[SEL_ROWS][32];
    const int k = blockIdx.x * 32 + threadIdx.x;
    const int f = blockIdx.y;
    const int64_t j0 = (int64_t)blockIdx.z * (SEL_ROWS * SEL_RPT);
    double m = 0.0;
    if (k < K) {
        const double* c = coef + (int64_t)f * p * ldz + k;
        for (int r = threadIdx.y; r < SEL_ROWS * SEL_RPT; r += SEL_ROWS) {
            const int64_t j = j0 + r;
            if (j < p) m = fmax(m, fabs(__ldg(c + j * ldz)));  // fmax drops a NaN operand
        }
    }
    part[threadIdx.y][threadIdx.x] = m;
    __syncthreads();
    if (threadIdx.y == 0 && k < K) {
#pragma unroll
        for (int r = 1; r < SEL_ROWS; ++r) m = fmax(m, part[r][threadIdx.x]);
        if (m > 0.0) atomicMax(colmax + (int64_t)f * ldz + k, (unsigned long long)__double_as_longlong(m));
    }
}

// Stage 2: one warp per feature j, lane = candidate column k (32 at a time).  Each thread adds the predicates of
// its (j, k) over the F fits of the chunk to counts[j][k] (one writer per entry: no atomics), and a ballot over
// the columns gives bit f of "feature j selected by some candidate of fit f", OR-ed into union[f][j].
__global__ void __launch_bounds__(32 * SEL_ROWS) support_count_kernel(const double* __restrict__ coef, int F,
                                                                      int64_t p, int64_t ldz, int K, double rel_tol,
                                                                      const unsigned long long* __restrict__ colmax,
                                                                      int32_t* __restrict__ counts,
                                                                      uint8_t* __restrict__ uni) {
    const int64_t j = (int64_t)blockIdx.x * SEL_ROWS + threadIdx.y;
    if (j >= p) return;  // whole warps leave: the ballots below see full warps
    const int lane = threadIdx.x;
    unsigned any = 0;  // bit f: feature j selected in fit f
    for (int k0 = 0; k0 < K; k0 += 32) {
        const int k = k0 + lane;
        int cnt = 0;
        for (int f = 0; f < F; ++f) {
            bool sel = false;
            if (k < K) {
                const double thr = rel_tol * __longlong_as_double((long long)__ldg(colmax + (int64_t)f * ldz + k));
                sel = fabs(__ldg(coef + ((int64_t)f * p + j) * ldz + k)) > thr;  // false for NaN
            }
            cnt += sel;
            if (__ballot_sync(0xffffffffu, sel)) any |= 1u << f;
        }
        if (k < K) counts[j * K + k] += cnt;
    }
    if (lane < F && ((any >> lane) & 1u)) uni[(int64_t)lane * p + j] = 1;
}

}  // namespace slm
