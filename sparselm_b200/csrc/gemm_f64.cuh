// FP64 tensor-core GEMM core for sm_100a (DMMA via mma.sync.m8n8k4.f64).
//
// FP64 has no tcgen05/UMMA kind on Blackwell, so the tensor path for doubles is
// warp-level mma.sync (SASS: DMMA.8x8x4) fed from shared memory; operands are
// staged global->shared with a multi-stage cp.async (LDGSTS) pipeline.
//
// One kernel serves every dense contraction of the hot path:
//   * Gram build   G_f = Xa_f^T Xa_f          (A K-major, symmetric: upper tiles + mirror)
//   * Gram apply   GZ_f = G_f Z_f             (A K-major through G's symmetry)
//   * CV scoring   Yhat_f = Xte_f B_f         (A M-major)
// i.e. C[M x N] = A[M x Kd] * B[Kd x N] with B row-major [Kd][ldq] and A given
// either as its transpose (row-major [Kd][ldp], "K-major") or row-major [M][ldp].
//
// Scheduling is data-parallel waves + stream-K over a persistent grid (SMs x CTAs/SM): as
// long as whole waves of tiles remain, CTA c takes tile c of the wave and runs its full
// contraction (all CTAs of a wave then sweep k in step and share operand panels through
// L2: one DRAM read of the operands per wave instead of one per tile); the (tile, k-slab)
// units of the partial last wave are laid out on one line and cut into equal contiguous
// ranges, one per CTA, so that the 148 SMs finish together whatever the tile count.  A CTA whose range covers a whole tile stores it.  A
// tile cut into several chunks is combined in a FIXED order (descending k: the
// chunk holding the tile's last slab stores, every earlier chunk waits on the
// tile's flag for the chunks after it and then adds), so results are
// bit-reproducible; the wait is short because in stream-K the later chunks of a
// tile are the ones that finish first.  All CTAs are co-resident (persistent
// grid), which makes the spin-wait safe.
//
// Row-sparse contraction (KSPARSE): the iterates of a sparse linear model are
// mostly exact zeros, so the apply only needs the rows k of Z (and the matching
// rows of G, by symmetry) where some column of the problem's column chunk is
// non-zero.  A problem then carries a device-side index list kidx[0..*kcount) of
// those rows; the contraction runs over the list (row gather in the cp.async
// loads) and, because the list length is only known on the device, every CTA
// derives the stream-K unit partition itself from the counts.
//
// Gathered Gram (SYM && KSPARSE): C = Xa[idx]^T Xa[idx] for a row list idx whose length is known on
// the host.  The contraction gathers rows as above, but the unit partition is the host-made hybrid
// one (data-parallel waves + stream-K remainder): the device-derived pure stream-K partition of the
// apply reads the operands once per tile instead of once per wave.
//
// Gathered A rows (AGATHER, A_MMAJOR only): row m of the M-major A operand is row kidx[m] of P
// (scoring of an arbitrary row set: predictions of the rows kidx[0..M)).
//
// Shared-memory tiles are padded by 4 doubles per row: for the m8n8k4 fragment
// pattern (k = lane%4, x = lane/4) a row stride == 4 or 12 (mod 16) doubles makes
// every half-warp hit 16 distinct 8-byte banks.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace slm {

constexpr int kMaxGemmProblems = 32;

struct GemmProblem {
    const double* P;  // A operand (see A_MMAJOR)
    const double* Q;  // B operand, row-major [Kd][ldq]
    double* C;        // row-major [M][ldc]
    const int* kidx;    // KSPARSE: rows of the contraction (ascending), else NULL
    const int* kcount;  // KSPARSE: device-side length of kidx
    long long ldp, ldq, ldc;
    int qlim;  // readable columns of a Q row from the Q pointer on (<= ldq)
    int M, N, Kd;
    int tiles_m, tiles_n;
    int n_tiles;     // tiles of this problem (upper triangle only when SYM)
    int kt;          // k-slabs per tile
    int unit_begin;  // first linear work unit (tile * kt + slab) of this problem
    int flag_begin;  // first per-tile flag of this problem
    int tile_begin;  // first global tile index of this problem
    // TMA kernels (gemm_f64_tma.cuh): the operands are addressed through tensor maps over the whole
    // matrices baseP / baseQ of the batch; a problem starts at these rows / this column of them
    int prow0, qrow0, qcol0, pcol0;
};

struct GemmBatch {
    int n_problems;
    int total_units;
    int units_per_cta;
    // hybrid schedule (host-partitioned batches): CTA c first computes the whole tiles
    // c, c + grid, ..., c + (full_waves-1)*grid ("data-parallel waves": every CTA walks the
    // contraction in step, so the operand panels of a wave are read from DRAM once and shared
    // through L2), then its stream-K share of the units from rem_unit_begin on (the partial
    // last wave, cut evenly so that all SMs finish together)
    int full_waves;
    int rem_unit_begin;
    int* flags;  // one int per tile, zero on entry
    int n_flags;
    int accumulate;  // != 0: C += A B (the tile's first writer adds to what C holds)
    int negate;      // != 0: the product enters with a minus sign (C -= A B with accumulate)
    int upper_only;  // SYM: only the tiles tn >= tm are written, no mirrored copy (blocked Cholesky)
    // TMA kernels: base matrices of the P / Q operands of every problem and their row counts
    // (NULL: the batch can only run on the cp.async kernel)
    const double *baseP, *baseQ;
    long long rowsP, rowsQ;
    GemmProblem pr[kMaxGemmProblems];
};

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile(
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    int bytes = valid ? 16 : 0;  // src-size 0 => 16 bytes of zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(gsrc), "r"(bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

template <int WARPS_M, int WARPS_N, int MI, int NI, int BK, int STAGES, bool A_MMAJOR>
struct GemmCfg {
    static constexpr int BM = WARPS_M * MI * 8;
    static constexpr int BN = WARPS_N * NI * 8;
    static constexpr int NT = WARPS_M * WARPS_N * 32;
    static constexpr int A_LD = A_MMAJOR ? (BK + 4) : (BM + 4);
    static constexpr int A_ROWS = A_MMAJOR ? BM : BK;
    static constexpr int B_LD = BN + 4;
    static constexpr int A_STAGE = A_ROWS * A_LD;  // doubles
    static constexpr int B_STAGE = BK * B_LD;
    static constexpr size_t SMEM = (size_t)STAGES * (A_STAGE + B_STAGE) * sizeof(double);
};

// SYM: problem is C = A^T A with P == Q; only tiles with tn >= tm exist and each
// is also written transposed.
template <int WARPS_M, int WARPS_N, int MI, int NI, int BK, int STAGES, bool A_MMAJOR, bool SYM, int MINB,
          bool KSPARSE = false, bool AGATHER = false>
__global__ void __launch_bounds__(WARPS_M* WARPS_N * 32, MINB)
    gemm_f64_kernel(const __grid_constant__ GemmBatch batch) {
    static_assert(!(KSPARSE && A_MMAJOR), "row-sparse mode is for the K-major contractions");
    static_assert(!AGATHER || (A_MMAJOR && !SYM && !KSPARSE), "gathered A rows are for the M-major scoring GEMM");
    // device-derived unit partition: the row-sparse apply, whose list lengths only the device knows
    constexpr bool DEV_PART = KSPARSE && !SYM;
    using Cfg = GemmCfg<WARPS_M, WARPS_N, MI, NI, BK, STAGES, A_MMAJOR>;
    constexpr int BM = Cfg::BM, BN = Cfg::BN, NT = Cfg::NT;
    extern __shared__ __align__(16) double smem[];
    double* As = smem;
    double* Bs = smem + (size_t)STAGES * Cfg::A_STAGE;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int lk = lane & 3, lx = lane >> 2;

    // unit partition: host-made, or derived here from the device-side row counts
    __shared__ int s_ub[DEV_PART ? kMaxGemmProblems + 1 : 1];
    __shared__ int s_kd[DEV_PART ? kMaxGemmProblems : 1];
    int upc = batch.units_per_cta, total_units = batch.total_units;
    if (DEV_PART) {
        if (tid < batch.n_problems) s_kd[tid] = min(batch.pr[tid].Kd, __ldcg(batch.pr[tid].kcount));
        __syncthreads();
        if (tid == 0) {
            int acc = 0;
            for (int i = 0; i < batch.n_problems; ++i) {
                s_ub[i] = acc;
                acc += batch.pr[i].n_tiles * max(1, (s_kd[i] + BK - 1) / BK);
            }
            s_ub[batch.n_problems] = acc;
        }
        __syncthreads();
        total_units = s_ub[batch.n_problems];
        upc = (total_units + (int)gridDim.x - 1) / (int)gridDim.x;
    }
    const int rem0 = DEV_PART ? 0 : batch.rem_unit_begin;  // first unit of the stream-K part
    int u = rem0 + blockIdx.x * upc;
    const int u_end = min(total_units, u + upc);
    int wave = 0;
    const int full_waves = DEV_PART ? 0 : batch.full_waves;

#pragma unroll 1
    while (wave < full_waves || u < u_end) {
        // ---- locate (problem, tile, slab range) of this segment ------------------
        int pi = 0, tl, kt0, kt1, KT, Kd, unit_begin;
        if (wave < full_waves) {  // a whole tile of a data-parallel wave
            const int tg = wave * (int)gridDim.x + (int)blockIdx.x;
            ++wave;
#pragma unroll 1
            for (int i = 1; i < batch.n_problems; ++i)
                if (tg >= batch.pr[i].tile_begin) pi = i;
            Kd = batch.pr[pi].Kd;
            KT = batch.pr[pi].kt;
            unit_begin = batch.pr[pi].unit_begin;
            tl = tg - batch.pr[pi].tile_begin;
            kt0 = 0;
            kt1 = KT;
        } else {
#pragma unroll 1
            for (int i = 1; i < batch.n_problems; ++i)
                if (u >= (DEV_PART ? s_ub[i] : batch.pr[i].unit_begin)) pi = i;
            Kd = DEV_PART ? s_kd[pi] : batch.pr[pi].Kd;
            KT = DEV_PART ? max(1, (Kd + BK - 1) / BK) : batch.pr[pi].kt;
            unit_begin = DEV_PART ? s_ub[pi] : batch.pr[pi].unit_begin;
            const int local = u - unit_begin;
            tl = local / KT;
            kt0 = local - tl * KT;
            kt1 = min(KT, kt0 + (u_end - u));
            u += kt1 - kt0;
        }
        const GemmProblem& pr = batch.pr[pi];
        const int tile_lin = tl;
        int tm, tn;
        if (SYM) {
            tm = 0;
            int rowlen = pr.tiles_n;
#pragma unroll 1
            while (tl >= rowlen) {
                tl -= rowlen;
                ++tm;
                --rowlen;
            }
            tn = tm + tl;
        } else {
            tm = tl / pr.tiles_n;
            tn = tl - tm * pr.tiles_n;
        }
        const int m0 = tm * BM, n0 = tn * BN;
        const int M = pr.M, N = pr.N, qlim = pr.qlim;
        const long long ldp = pr.ldp, ldq = pr.ldq, ldc = pr.ldc;
        const double* __restrict__ P = pr.P;
        const double* __restrict__ Q = pr.Q;
        const int* __restrict__ kidx = pr.kidx;

        double acc[MI][NI][2];
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
            for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        if (batch.accumulate) {
            // the tile of the accumulated-into matrix is wanted in the epilogue: start bringing it to L2 now
#pragma unroll
            for (int i = 0; i < MI; ++i)
#pragma unroll
                for (int j = 0; j < NI; ++j) {
                    const int row = m0 + (wm * MI + i) * 8 + lx, col = n0 + (wn * NI + j) * 8 + lk * 2;
                    if (row < M && col < N)
                        asm volatile("prefetch.global.L2 [%0];\n" ::"l"(pr.C + (long long)row * ldc + col));
                }
        }

        // KSPARSE: the gathered row index of every 16-byte chunk this thread copies is
        // fetched one slab ahead into registers (pidx_*), so the dependent index -> cp.async
        // chain never sits on the critical path of the slab loop
        constexpr int A_CPR = A_MMAJOR ? BK / 2 : BM / 2;  // 16-byte chunks per A tile row
        constexpr int B_CPR = BN / 2;
        constexpr int A_IT = (BK * A_CPR + NT - 1) / NT;
        constexpr int B_IT = (BK * B_CPR + NT - 1) / NT;
        int pidx_a[KSPARSE ? A_IT : 1], pidx_b[KSPARSE ? B_IT : 1];
        auto fetch_idx = [&](int kt) {  // indices of slab kt (or -1: zero fill)
            const int k0 = kt * BK;
#pragma unroll
            for (int i = 0; i < A_IT; ++i) {
                const int c = tid + i * NT, r = c / A_CPR;
                pidx_a[i] = (c < BK * A_CPR && k0 + r < Kd) ? __ldg(kidx + k0 + r) : -1;
            }
#pragma unroll
            for (int i = 0; i < B_IT; ++i) {
                const int c = tid + i * NT, r = c / B_CPR;
                pidx_b[i] = (c < BK * B_CPR && k0 + r < Kd) ? __ldg(kidx + k0 + r) : -1;
            }
        };
        auto load_stage_sparse = [&](int stage) {  // slab described by pidx_*
            double* as = As + (size_t)stage * Cfg::A_STAGE;
            double* bs = Bs + (size_t)stage * Cfg::B_STAGE;
#pragma unroll
            for (int i = 0; i < A_IT; ++i) {
                const int c = tid + i * NT;
                if (c < BK * A_CPR) {
                    const int r = c / A_CPR, x = (c - r * A_CPR) * 2;
                    const long long col = (long long)m0 + x;
                    const bool ok = pidx_a[i] >= 0 && (col + 2 <= ldp);
                    const double* src = ok ? (P + (long long)pidx_a[i] * ldp + col) : P;
                    cp_async16(as + r * Cfg::A_LD + x, src, ok);
                }
            }
#pragma unroll
            for (int i = 0; i < B_IT; ++i) {
                const int c = tid + i * NT;
                if (c < BK * B_CPR) {
                    const int r = c / B_CPR, x = (c - r * B_CPR) * 2;
                    const long long col = (long long)n0 + x;
                    const bool ok = pidx_b[i] >= 0 && (col + 2 <= qlim);
                    const double* src = ok ? (Q + (long long)pidx_b[i] * ldq + col) : Q;
                    cp_async16(bs + r * Cfg::B_LD + x, src, ok);
                }
            }
        };
        // AGATHER: the source rows of the A tile are the same for every slab of the tile
        constexpr int AG_IT = AGATHER ? (BM * (BK / 2) + NT - 1) / NT : 1;
        long long arow[AG_IT];
        if (AGATHER) {
#pragma unroll
            for (int i = 0; i < AG_IT; ++i) {
                const int r = (tid + i * NT) / (BK / 2);
                arow[i] = (r < BM && m0 + r < M) ? (long long)__ldg(kidx + m0 + r) : -1;
            }
        }
        auto load_stage = [&](int kt, int stage) {
            const int k0 = kt * BK;
            double* as = As + (size_t)stage * Cfg::A_STAGE;
            double* bs = Bs + (size_t)stage * Cfg::B_STAGE;
            if (AGATHER) {
                constexpr int CPR = BK / 2;
#pragma unroll
                for (int i = 0; i < AG_IT; ++i) {
                    const int c = tid + i * NT;
                    if (c < BM * CPR) {
                        const int r = c / CPR, x = (c - r * CPR) * 2;
                        const bool ok = arow[i] >= 0 && (k0 + x + 2 <= ldp);
                        const double* src = ok ? (P + arow[i] * ldp + k0 + x) : P;
                        cp_async16(as + r * Cfg::A_LD + x, src, ok);
                    }
                }
            } else if (!A_MMAJOR) {
                constexpr int CPR = BM / 2;  // 16-byte chunks per row
                for (int c = tid; c < BK * CPR; c += NT) {
                    int r = c / CPR, x = (c - r * CPR) * 2;
                    long long col = (long long)m0 + x;
                    bool ok = (k0 + r < Kd) && (col + 2 <= ldp);
                    const double* src = ok ? (P + (long long)(k0 + r) * ldp + col) : P;
                    cp_async16(as + r * Cfg::A_LD + x, src, ok);
                }
            } else {
                constexpr int CPR = BK / 2;
                for (int c = tid; c < BM * CPR; c += NT) {
                    int r = c / CPR, x = (c - r * CPR) * 2;
                    // columns >= Kd (inside the row allocation) may be loaded: the matching
                    // rows of the B tile are zero-filled, and Xa's padding is finite
                    bool ok = (m0 + r < M) && (k0 + x + 2 <= ldp);
                    const double* src = ok ? (P + (long long)(m0 + r) * ldp + k0 + x) : P;
                    cp_async16(as + r * Cfg::A_LD + x, src, ok);
                }
            }
            {
                constexpr int CPR = BN / 2;
                for (int c = tid; c < BK * CPR; c += NT) {
                    int r = c / CPR, x = (c - r * CPR) * 2;
                    long long col = (long long)n0 + x;
                    bool ok = (k0 + r < Kd) && (col + 2 <= qlim);
                    const double* src = ok ? (Q + (long long)(k0 + r) * ldq + col) : Q;
                    cp_async16(bs + r * Cfg::B_LD + x, src, ok);
                }
            }
        };

        // ---- prologue ------------------------------------------------------------
        const int nkt = kt1 - kt0;
#pragma unroll
        for (int s = 0; s < STAGES - 1; ++s) {
            if (s < nkt) {
                if (KSPARSE) {
                    fetch_idx(kt0 + s);
                    load_stage_sparse(s);
                } else {
                    load_stage(kt0 + s, s);
                }
            }
            cp_async_commit();
        }
        if (KSPARSE && STAGES - 1 < nkt) fetch_idx(kt0 + STAGES - 1);

        // ---- main loop -----------------------------------------------------------
#pragma unroll 1
        for (int it = 0; it < nkt; ++it) {
            cp_async_wait<STAGES - 2>();
            __syncthreads();
            {
                int nk = it + STAGES - 1;
                if (nk < nkt) {
                    if (KSPARSE) {
                        load_stage_sparse(nk % STAGES);
                        if (nk + 1 < nkt) fetch_idx(kt0 + nk + 1);  // consumed by the next iteration
                    } else {
                        load_stage(kt0 + nk, nk % STAGES);
                    }
                }
                cp_async_commit();
            }
            const double* as = As + (size_t)(it % STAGES) * Cfg::A_STAGE;
            const double* bs = Bs + (size_t)(it % STAGES) * Cfg::B_STAGE;
#pragma unroll
            for (int kk = 0; kk < BK / 4; ++kk) {
                double a[MI], b[NI];
#pragma unroll
                for (int i = 0; i < MI; ++i) {
                    int m = (wm * MI + i) * 8 + lx;
                    a[i] = A_MMAJOR ? as[m * Cfg::A_LD + kk * 4 + lk] : as[(kk * 4 + lk) * Cfg::A_LD + m];
                }
#pragma unroll
                for (int j = 0; j < NI; ++j) {
                    int n = (wn * NI + j) * 8 + lx;
                    b[j] = bs[(kk * 4 + lk) * Cfg::B_LD + n];
                }
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int j = 0; j < NI; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();  // smem is reused by the next segment

        // ---- epilogue --------------------------------------------------------------
        double* __restrict__ C = pr.C;
        const bool whole = (kt0 == 0) && (kt1 == KT);
        const bool first_writer = (kt1 == KT);  // holds the tile's last slab: stores
        int* flag = batch.flags + pr.flag_begin + tile_lin;
        if (!whole && !first_writer) {
            // chunks after mine = CTAs between me and the one owning the tile's last unit
            const int tile_last_unit = unit_begin + tile_lin * KT + KT - 1;
            const int after = (tile_last_unit - rem0) / upc - (int)blockIdx.x;
            if (tid == 0) {
                while (atomicAdd(flag, 0) < after) __nanosleep(64);
                __threadfence();
            }
            __syncthreads();
        }
        // the earlier partial sum / the accumulated-into matrix is read in batches of one row block (NI
        // independent loads in flight) BEFORE any store of that block: written load-add-store element by
        // element, every load waits behind the previous store (the compiler cannot reorder them: the pointers
        // may alias) and the epilogue costs MI * NI serialised memory round trips
        const bool need_old = !first_writer || batch.accumulate;
        constexpr int JB = NI < 4 ? NI : 4;  // loads in flight per batch (more would cost registers the main loop needs)
#pragma unroll
        for (int i = 0; i < MI; ++i) {
            const int row = m0 + (wm * MI + i) * 8 + lx;
#pragma unroll
            for (int j0 = 0; j0 < NI; j0 += JB) {
                double2 old[JB];
#pragma unroll
                for (int jj = 0; jj < JB; ++jj) {
                    const int col = n0 + (wn * NI + j0 + jj) * 8 + lk * 2;
                    old[jj] = make_double2(0.0, 0.0);
                    if (j0 + jj < NI && need_old && row < M && col < N)
                        old[jj] = __ldcg(reinterpret_cast<const double2*>(C + (long long)row * ldc + col));
                }
#pragma unroll
                for (int jj = 0; jj < JB; ++jj) {
                    const int j = j0 + jj;
                    const int col = n0 + (wn * NI + j) * 8 + lk * 2;
                    if (j < NI && row < M && col < N) {  // N is even: col+1 < N too
                        double v0 = acc[i][j < NI ? j : 0][0], v1 = acc[i][j < NI ? j : 0][1];
                        if (batch.negate) {
                            v0 = -v0;
                            v1 = -v1;
                        }
                        v0 += old[jj].x;
                        v1 += old[jj].y;
                        double2* dst = reinterpret_cast<double2*>(C + (long long)row * ldc + col);
                        __stcg(dst, make_double2(v0, v1));
                        if (SYM && tm != tn && !batch.upper_only) {
                            // mirrored copy: same value as the upper entry (kept bit-identical)
                            __stcg(C + (long long)col * ldc + row, v0);
                            __stcg(C + (long long)(col + 1) * ldc + row, v1);
                        }
                    }
                }
            }
        }
        if (!whole) {
            __threadfence();
            __syncthreads();
            if (tid == 0) atomicAdd(flag, 1);
        }
    }
}

}  // namespace slm
