// Stability selection: selection counts of the coefficient tables of one chunk of subsample fits per feature
// (slm_support_counts) and per group (slm_group_support_counts), and the random column weights of randomized
// stability selection applied to the chunk's training Grams (slm_gram_scale); DESIGN section 2 item 17.
//
// coef is [F][p][ldz] as the solve returns it (fit f, feature j, candidate column k).  Coefficient j of
// fit (f, k) is selected iff |coef| > rel_tol * max_j' |coef[f][j'][k]|; an all-zero fit selects nothing
// and a NaN coefficient is never selected.  Columns k >= K (batch padding) are never read.  A group is
// selected in a fit iff one of its features is.
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

// Stage 2 of the group counts: one block per group g (features gptr[g] .. gptr[g+1]), lane = candidate column k
// (32 at a time).  The block's warps stride over the group's features, so a group of any length from 1 to p is
// read by all SEL_ROWS warps; each thread keeps bit f of "some feature of g in its rows selected for (f, k)" and
// the warps' masks are OR-ed in shared memory.  Thread (warp 0, lane) then adds the popcount of the merged mask
// to counts[g][k] (one writer per entry: no atomics), and an OR over the lanes gives bit f of "g selected by some
// candidate of fit f", OR-ed into union[f][g].  The predicate of one feature is the one of support_count_kernel.
__global__ void __launch_bounds__(32 * SEL_ROWS) group_support_count_kernel(
    const double* __restrict__ coef, int F, int64_t p, int64_t ldz, int K, double rel_tol,
    const unsigned long long* __restrict__ colmax, const int32_t* __restrict__ gptr, int n_groups,
    int32_t* __restrict__ counts, uint8_t* __restrict__ uni) {
    __shared__ unsigned part[SEL_ROWS][32];
    const int g = blockIdx.x;
    const int lane = threadIdx.x;
    const int64_t j0 = __ldg(gptr + g), j1 = __ldg(gptr + g + 1);
    unsigned any = 0;  // warp 0: bit f, g selected by some candidate of fit f
    for (int k0 = 0; k0 < K; k0 += 32) {
        const int k = k0 + lane;
        unsigned m = 0;
        if (k < K) {
            for (int f = 0; f < F; ++f) {
                const double thr = rel_tol * __longlong_as_double((long long)__ldg(colmax + (int64_t)f * ldz + k));
                const double* c = coef + (int64_t)f * p * ldz + k;
                bool sel = false;
                for (int64_t j = j0 + threadIdx.y; j < j1; j += SEL_ROWS)
                    sel |= fabs(__ldg(c + j * ldz)) > thr;  // false for NaN
                m |= (unsigned)sel << f;
            }
        }
        part[threadIdx.y][lane] = m;
        __syncthreads();
        if (threadIdx.y == 0) {
#pragma unroll
            for (int r = 1; r < SEL_ROWS; ++r) m |= part[r][lane];
            if (k < K) counts[(int64_t)g * K + k] += __popc(m);
            any |= __reduce_or_sync(0xffffffffu, m);
        }
        __syncthreads();  // part is rewritten by the next column chunk
    }
    if (threadIdx.y == 0 && lane < F && ((any >> lane) & 1u)) uni[(int64_t)lane * n_groups + g] = 1;
}

// Randomized stability selection (slm_gram_scale): G[s][i][j] *= d_i * d_j in place, d_i = w[slot[s]][i] for
// i < p and 1 for the y row, the ones row and the padding.  One block per (row i, Gram s); the product d_i * d_j
// is rounded once and then multiplies G, which is bitwise numpy's G * np.outer(d, d) and keeps G exactly
// symmetric.  Rows i >= p only scale their first p columns; nothing in the trailing block is touched.
struct GramScaleSlots {
    int32_t slot[16];  // SLM_MAX_FOLDS: row of the weights table of Gram s
};

__global__ void __launch_bounds__(256) gram_scale_kernel(double* __restrict__ G, int64_t g_stride, int64_t pa,
                                                         int64_t p, const double* __restrict__ w, GramScaleSlots sl) {
    const int64_t i = blockIdx.x;
    const int s = blockIdx.y;
    const double* ws = w + (int64_t)sl.slot[s] * p;
    const double di = i < p ? __ldg(ws + i) : 1.0;
    double* row = G + (int64_t)s * g_stride + i * pa;
    const int64_t jend = i < p ? pa : p;
    for (int64_t j = threadIdx.x; j < jend; j += blockDim.x) {
        const double dj = j < p ? __ldg(ws + j) : 1.0;
        row[j] = row[j] * __dmul_rn(di, dj);
    }
}

}  // namespace slm
