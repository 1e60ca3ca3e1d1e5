// TMA-fed FP64 tensor-core GEMM for sm_100a: cp.async.bulk.tensor (tiled and tile::gather4) +
// mbarrier producer/consumer ring + DMMA (mma.sync.m8n8k4.f64) consumers.
//
// Same contraction, scheduling (data-parallel waves + stream-K remainder, fixed-order fix-up,
// device-derived unit partition for the row-sparse mode) and epilogue as gemm_f64.cuh; what
// changes is how the operand tiles reach shared memory.  In the cp.async kernel every compute
// thread issues its share of the 16-byte copies of a k-slab (address arithmetic, predicates,
// index gathers: ~3x the issue slots of the slab's DMMAs, with the DMMA pipe idle behind the
// CTA-wide barrier).  Here ONE extra warp is the producer: it waits for a free stage, arms the
// stage's mbarrier with the byte count and issues a handful of TMA operations -- 2-D boxes of
// [BK rows x 16 doubles] for the dense contractions, tile::gather4 row gathers (4 arbitrary rows
// x 16 doubles per operation, row indices straight from the device-side support list) for the
// row-sparse Gram apply.  The consumer warps only wait on the stage's mbarrier, read fragments
// and issue DMMAs; there is no __syncthreads in the main loop.
//
// Shared-memory layout: every operand tile is a row of boxes, a box is [BK][16 doubles] = BK
// rows of 128 bytes written by the TMA unit with the 128-byte swizzle (16-byte chunk index XOR
// (row & 7)).  The m8n8k4 fragment of lane (lk = lane & 3, lx = lane >> 2) is element
// (k = lk, x = lx); a dense row stride of 128 bytes would put the four k rows of a fragment on
// the same banks, so the contraction index is permuted inside every group of 8 slab rows:
// k-step 2t uses rows 8t + {0, 2, 4, 6}, k-step 2t+1 rows 8t + {1, 3, 5, 7} (the same
// permutation for both operands, so the product is unchanged).  Rows of equal parity have
// (row & 7) in {0,2,4,6} or {1,3,5,7}: the XOR then maps the two chunks a half-warp touches per
// row to four disjoint chunk pairs -- 16 distinct 8-byte banks, conflict-free without padding.
//
// WIDE layout (template flag): one TMA operation moves a tile row band of BM+4 (BN+4) doubles
// WITHOUT swizzle -- rows of (BM+4)*8 bytes, a pitch that is 32 (or 96) mod 128 bytes, so the four k rows of
// a fragment fall on four different 32-byte bank groups (the same padded layout as the cp.async kernel,
// written by the TMA unit).  A k-slab then takes 2 operations (tiled) or 2 per four gathered rows instead
// of one per 128-byte box: the row-sparse apply at 32-column tiles issued 40 gather operations of 512 bytes
// per slab and ran at the TMA unit's operation rate (about one per 46 cycles per SM = 3.1 TB/s), not at the
// DMMA rate.
//
// Tails.  Rows of the last k-slab beyond the contraction length are not masked by the copy
// (dense: they are the next rows of the matrix or zero-filled out-of-bounds rows; gather: the
// list is padded with its last index): the consumers zero both fragments of those rows.  Columns
// beyond the matrix are zero-filled by the TMA unit; columns beyond a problem's N are computed
// and never stored.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm_f64.cuh"

namespace slm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// 2-D tiled load: box (c0 = first column, c1 = first row) of the tensor map into smem
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
        "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// row gather: rows r0..r3 (arbitrary) x one box width of columns starting at c0
__device__ __forceinline__ void tma_gather4(uint32_t dst, const CUtensorMap* map, int c0, int r0, int r1, int r2, int r3,
                                            uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];\n" ::
            "r"(dst),
        "l"(map), "r"(c0), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar)
        : "memory");
}
constexpr int kTmaBoxCols = 16;  // doubles per box row = 128 bytes (the swizzle span)

template <int WARPS_M, int WARPS_N, int MI, int NI, int BK, int STAGES, bool WIDE>
struct TmaCfg {
    static constexpr int BM = WARPS_M * MI * 8;
    static constexpr int BN = WARPS_N * NI * 8;
    static constexpr int NCW = WARPS_M * WARPS_N;       // consumer warps
    // + one producer warp GROUP: register re-allocation (setmaxnreg) works on groups of four
    // warps, and so does the register file's allocation quantum -- a single extra warp would
    // cost the same registers.  Only the first warp of the group issues copies.
    static constexpr int NT = (NCW + 4) * 32;
    static_assert(NCW % 4 == 0, "consumer warps come in groups of four (setmaxnreg)");
    // swizzled layout: boxes of [BK][16 doubles]
    static constexpr int ABOX = BM / kTmaBoxCols;
    static constexpr int BBOX = (BN + kTmaBoxCols - 1) / kTmaBoxCols;
    static constexpr int BOXB = BK * 128;                // bytes per box
    // wide layout: one band of BM+4 / BN+4 doubles per row
    static constexpr int A_COLS = WIDE ? BM + 4 : kTmaBoxCols;  // box width of the P map (doubles)
    static constexpr int B_COLS = WIDE ? BN + 4 : kTmaBoxCols;
    static constexpr int A_PITCH = (BM + 4) * 8, B_PITCH = (BN + 4) * 8;  // bytes (WIDE)
    static constexpr int A_BYTES = WIDE ? BK * A_PITCH : ABOX * BOXB;
    static constexpr int STAGE_BYTES = WIDE ? BK * (A_PITCH + B_PITCH) : (ABOX + BBOX) * BOXB;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 2 * STAGES * 8 + 64;
    static_assert(BM % kTmaBoxCols == 0, "the M tile must be whole boxes");
    static_assert(BK % 8 == 0, "slabs are groups of 8 rows (swizzle period)");
    static_assert(A_BYTES % 128 == 0 && STAGE_BYTES % 128 == 0, "TMA destinations are 128-byte aligned");
};

// A operand K-major only (Gram build, Gram apply).  SYM / KSPARSE as in gemm_f64_kernel (SYM && KSPARSE:
// the gathered Gram, host-made hybrid partition).
// mapP / mapQ: 2-D tensor maps over the whole operand matrices (P: [rows][ldp], Q: [rows][ldq]),
// box [BK][16] for the tiled mode, [1][16] for the gather mode.  A problem addresses its rows
// through prow0 / qrow0 and its first P / Q columns through pcol0 / qcol0.
template <int WARPS_M, int WARPS_N, int MI, int NI, int BK, int STAGES, bool SYM, int MINB, bool KSPARSE, bool WIDE>
__global__ void __launch_bounds__((WARPS_M * WARPS_N + 4) * 32, MINB)
    gemm_f64_tma_kernel(const __grid_constant__ GemmBatch batch, const __grid_constant__ CUtensorMap mapP,
                        const __grid_constant__ CUtensorMap mapQ) {
    using Cfg = TmaCfg<WARPS_M, WARPS_N, MI, NI, BK, STAGES, WIDE>;
    constexpr int BM = Cfg::BM, BN = Cfg::BN, NCW = Cfg::NCW;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t tiles0 = (smem_u32(smem_raw) + 1023u) & ~1023u;  // 1024-byte aligned: swizzle atoms
    const uint8_t* tiles_ptr = smem_raw + (tiles0 - smem_u32(smem_raw));
    const uint32_t bars0 = tiles0 + (uint32_t)STAGES * Cfg::STAGE_BYTES;
    auto full_bar = [&](int s) { return bars0 + 8u * (uint32_t)s; };
    auto empty_bar = [&](int s) { return bars0 + 8u * (uint32_t)(STAGES + s); };

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // unit partition: host-made, or derived here from the device-side row counts (row-sparse apply)
    constexpr bool DEV_PART = KSPARSE && !SYM;
    __shared__ int s_ub[DEV_PART ? kMaxGemmProblems + 1 : 1];
    __shared__ int s_kd[DEV_PART ? kMaxGemmProblems : 1];
    int upc = batch.units_per_cta, total_units = batch.total_units;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), NCW);
        }
        mbar_fence_init();
    }
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
    }
    __syncthreads();
    if (DEV_PART) {
        total_units = s_ub[batch.n_problems];
        upc = (total_units + (int)gridDim.x - 1) / (int)gridDim.x;
    }
    const int rem0 = DEV_PART ? 0 : batch.rem_unit_begin;
    int u = rem0 + blockIdx.x * upc;
    const int u_end = min(total_units, u + upc);
    int wave = 0;
    const int full_waves = DEV_PART ? 0 : batch.full_waves;

    // (problem, tile, slab range) of the next segment of this CTA -- walked identically by the
    // producer warp and by the consumer warps
    struct Seg {
        int pi, tl, kt0, kt1, KT, Kd, unit_begin;
    };
    auto next_seg = [&](Seg& sg) -> bool {
        if (!(wave < full_waves || u < u_end)) return false;
        int pi = 0;
        if (wave < full_waves) {
            const int tg = wave * (int)gridDim.x + (int)blockIdx.x;
            ++wave;
#pragma unroll 1
            for (int i = 1; i < batch.n_problems; ++i)
                if (tg >= batch.pr[i].tile_begin) pi = i;
            sg.Kd = batch.pr[pi].Kd;
            sg.KT = batch.pr[pi].kt;
            sg.unit_begin = batch.pr[pi].unit_begin;
            sg.tl = tg - batch.pr[pi].tile_begin;
            sg.kt0 = 0;
            sg.kt1 = sg.KT;
        } else {
#pragma unroll 1
            for (int i = 1; i < batch.n_problems; ++i)
                if (u >= (DEV_PART ? s_ub[i] : batch.pr[i].unit_begin)) pi = i;
            sg.Kd = DEV_PART ? s_kd[pi] : batch.pr[pi].Kd;
            sg.KT = DEV_PART ? max(1, (sg.Kd + BK - 1) / BK) : batch.pr[pi].kt;
            sg.unit_begin = DEV_PART ? s_ub[pi] : batch.pr[pi].unit_begin;
            const int local = u - sg.unit_begin;
            sg.tl = local / sg.KT;
            sg.kt0 = local - sg.tl * sg.KT;
            sg.kt1 = min(sg.KT, sg.kt0 + (u_end - u));
            u += sg.kt1 - sg.kt0;
        }
        sg.pi = pi;
        return true;
    };
    auto tile_coords = [&](const GemmProblem& pr, int tl, int& tm, int& tn) {
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
    };

    uint32_t it_global = 0;  // slabs this CTA has gone through: stage = it % STAGES, phase from it / STAGES

    // register budget: the kernel starts with R0 registers per thread (what the launch bounds allow);
    // the producer group gives back all but PR, the consumer groups take their share of those
    constexpr int R0 = (65536 / (MINB * Cfg::NT)) / 8 * 8;
    constexpr int PR = 24;
    constexpr int CR_RAW = (R0 + (R0 - PR) * 4 / NCW) / 8 * 8;
    constexpr int CR = CR_RAW > 232 ? 232 : CR_RAW;

    if (warp >= NCW) {
        // ======================= producer warp group =======================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" ::"n"(PR));
        if (warp != NCW) return;
        Seg sg;
        while (next_seg(sg)) {
            const GemmProblem& pr = batch.pr[sg.pi];
            int tm, tn;
            tile_coords(pr, sg.tl, tm, tn);
            const int m0 = pr.pcol0 + tm * BM, n0 = pr.qcol0 + tn * BN;
            const int prow0 = pr.prow0, qrow0 = pr.qrow0;
            const int* __restrict__ kidx = pr.kidx;
#pragma unroll 1
            for (int kt = sg.kt0; kt < sg.kt1; ++kt, ++it_global) {
                const int stage = (int)(it_global % STAGES);
                const uint32_t phase = (it_global / STAGES) & 1u;
                mbar_wait(empty_bar(stage), phase ^ 1u);  // passes at once on a never-used stage
                const uint32_t sA = tiles0 + (uint32_t)stage * Cfg::STAGE_BYTES;
                const uint32_t sB = sA + Cfg::A_BYTES;
                const uint32_t fb = full_bar(stage);
                if (lane == 0) mbar_arrive_expect_tx(fb, Cfg::STAGE_BYTES);
                __syncwarp();
                const int k0 = kt * BK;
                if (!KSPARSE && WIDE) {
                    // one operation per operand: the whole [BK][BM+4] / [BK][BN+4] band of the slab
                    if (lane == 0) tma_load_2d(sA, &mapP, m0, prow0 + k0, fb);
                    if (lane == 1) tma_load_2d(sB, &mapQ, n0, qrow0 + k0, fb);
                } else if (!KSPARSE) {
                    // one box per lane round: boxes 0..ABOX-1 of A, then BBOX boxes of B
                    for (int b = lane; b < Cfg::ABOX + Cfg::BBOX; b += 32) {
                        if (b < Cfg::ABOX)
                            tma_load_2d(sA + (uint32_t)b * Cfg::BOXB, &mapP, m0 + b * kTmaBoxCols, prow0 + k0, fb);
                        else
                            tma_load_2d(sB + (uint32_t)(b - Cfg::ABOX) * Cfg::BOXB, &mapQ,
                                        n0 + (b - Cfg::ABOX) * kTmaBoxCols, qrow0 + k0, fb);
                    }
                } else {
                    // lane l holds the index of slab row l (lists are padded with their last entry,
                    // or row 0 when empty: the consumers zero the fragments of padded rows)
                    const int last = sg.Kd > 0 ? sg.Kd - 1 : -1;
                    int myidx = 0;
                    if (lane < BK) {
                        const int kk = min(k0 + lane, last);
                        myidx = kk >= 0 ? __ldg(kidx + kk) : 0;
                    }
                    constexpr int QUADS = BK / 4;
                    if (WIDE) {
                        // lane 2q gathers rows 4q..4q+3 of the A band, lane 2q+1 those of the B band
                        const int oq = min(lane >> 1, QUADS - 1);
                        const int r0 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 0);
                        const int r1 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 1);
                        const int r2 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 2);
                        const int r3 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 3);
                        if (lane < 2 * QUADS) {
                            if ((lane & 1) == 0)
                                tma_gather4(sA + (uint32_t)oq * 4u * Cfg::A_PITCH, &mapP, m0, prow0 + r0, prow0 + r1,
                                            prow0 + r2, prow0 + r3, fb);
                            else
                                tma_gather4(sB + (uint32_t)oq * 4u * Cfg::B_PITCH, &mapQ, n0, qrow0 + r0, qrow0 + r1,
                                            qrow0 + r2, qrow0 + r3, fb);
                        }
                        __syncwarp();
                        continue;
                    }
                    constexpr int OPS = QUADS * (Cfg::ABOX + Cfg::BBOX);
#pragma unroll 1
                    for (int o0 = 0; o0 < OPS; o0 += 32) {
                        const int o = o0 + lane;
                        const int oq = min(o, OPS - 1) / (Cfg::ABOX + Cfg::BBOX);
                        const int ob = min(o, OPS - 1) - oq * (Cfg::ABOX + Cfg::BBOX);
                        const int r0 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 0);
                        const int r1 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 1);
                        const int r2 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 2);
                        const int r3 = __shfl_sync(0xffffffffu, myidx, 4 * oq + 3);
                        if (o < OPS) {
                            if (ob < Cfg::ABOX)
                                tma_gather4(sA + (uint32_t)ob * Cfg::BOXB + (uint32_t)oq * 512u, &mapP,
                                            m0 + ob * kTmaBoxCols, prow0 + r0, prow0 + r1, prow0 + r2, prow0 + r3, fb);
                            else
                                tma_gather4(sB + (uint32_t)(ob - Cfg::ABOX) * Cfg::BOXB + (uint32_t)oq * 512u, &mapQ,
                                            n0 + (ob - Cfg::ABOX) * kTmaBoxCols, qrow0 + r0, qrow0 + r1, qrow0 + r2,
                                            qrow0 + r3, fb);
                        }
                    }
                }
                __syncwarp();
            }
        }
        return;
    }

    // ======================= consumer warps =======================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" ::"n"(CR));
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int lk = lane & 3, lx = lane >> 2;
    // byte offset of this lane's fragment element inside a stage for k-step 0 (rows 2*lk of the
    // first 8-row group); k-step j adds (j >> 1) * 1024 + (j & 1) * 128 and flips bit 4 when j is odd
    // The 8-column block t8 = w * XI + i of a lane's fragment i selects the box t8 >> 1 and the
    // half (t8 & 1) of its 128-byte rows.  For every tile shape in use the parity of t8 is known at
    // compile time (XI even, or a single warp along that dimension), so a lane needs two base
    // offsets per operand (one per half) and compile-time box strides on top of them.
    constexpr bool A_STATIC = (MI % 2 == 0) || (WARPS_M == 1);
    constexpr bool B_STATIC = (NI % 2 == 0) || (WARPS_N == 1);
    auto lane_off = [&](int half) {
        const int chunk = (half << 2) + (lx >> 1);
        return (uint32_t)lk * 256u + (uint32_t)((chunk ^ (2 * lk)) << 4) + (uint32_t)(lx & 1) * 8u;
    };
    const uint32_t laneoff[2] = {lane_off(0), lane_off(1)};
    const uint32_t wbaseA = A_STATIC ? (uint32_t)(wm * (MI / 2)) * Cfg::BOXB : 0u;  // MI odd: WARPS_M == 1, wm == 0
    const uint32_t wbaseB = Cfg::A_BYTES + (B_STATIC ? (uint32_t)(wn * (NI / 2)) * Cfg::BOXB : 0u);
    auto off_a = [&](int i) -> uint32_t {
        if (A_STATIC) return wbaseA + laneoff[i & 1] + (uint32_t)(i >> 1) * Cfg::BOXB;
        const int t8 = wm * MI + i;
        return (uint32_t)(t8 >> 1) * Cfg::BOXB + laneoff[t8 & 1];
    };
    auto off_b = [&](int j) -> uint32_t {
        if (B_STATIC) return wbaseB + laneoff[j & 1] + (uint32_t)(j >> 1) * Cfg::BOXB;
        const int t8 = wn * NI + j;
        return Cfg::A_BYTES + (uint32_t)(t8 >> 1) * Cfg::BOXB + laneoff[t8 & 1];
    };

    Seg sg;
#pragma unroll 1
    while (next_seg(sg)) {
        const GemmProblem& pr = batch.pr[sg.pi];
        const int tile_lin = sg.tl;
        int tm, tn;
        tile_coords(pr, sg.tl, tm, tn);
        const int m0 = tm * BM, n0 = tn * BN;
        const int M = pr.M, N = pr.N;
        const long long ldc = pr.ldc;

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

#pragma unroll 1
        for (int kt = sg.kt0; kt < sg.kt1; ++kt, ++it_global) {
            const int stage = (int)(it_global % STAGES);
            const uint32_t phase = (it_global / STAGES) & 1u;
            const uint8_t* sbase = tiles_ptr + (size_t)stage * Cfg::STAGE_BYTES;
            const int kd_rem = sg.Kd - kt * BK;  // valid rows of this slab (>= BK: all)
            mbar_wait(full_bar(stage), phase);
            if (WIDE) {
                // padded-pitch layout: element (k, x) of a band at k * PITCH + 8 x, natural k order
                const double* As = reinterpret_cast<const double*>(sbase);
                const double* Bs = reinterpret_cast<const double*>(sbase + Cfg::A_BYTES);
                constexpr int A_LD = BM + 4, B_LD = BN + 4;
                if (kd_rem >= BK) {
#pragma unroll
                    for (int s = 0; s < BK / 4; ++s) {
                        double a[MI], b[NI];
#pragma unroll
                        for (int i = 0; i < MI; ++i) a[i] = As[(s * 4 + lk) * A_LD + (wm * MI + i) * 8 + lx];
#pragma unroll
                        for (int j = 0; j < NI; ++j) b[j] = Bs[(s * 4 + lk) * B_LD + (wn * NI + j) * 8 + lx];
#pragma unroll
                        for (int i = 0; i < MI; ++i)
#pragma unroll
                            for (int j = 0; j < NI; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                    }
                } else {
#pragma unroll 1
                    for (int s = 0; s < BK / 4; ++s) {
                        const bool ok = s * 4 + lk < kd_rem;
                        double a[MI], b[NI];
#pragma unroll
                        for (int i = 0; i < MI; ++i) {
                            const double v = As[(s * 4 + lk) * A_LD + (wm * MI + i) * 8 + lx];
                            a[i] = ok ? v : 0.0;
                        }
#pragma unroll
                        for (int j = 0; j < NI; ++j) {
                            const double v = Bs[(s * 4 + lk) * B_LD + (wn * NI + j) * 8 + lx];
                            b[j] = ok ? v : 0.0;
                        }
#pragma unroll
                        for (int i = 0; i < MI; ++i)
#pragma unroll
                            for (int j = 0; j < NI; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                    }
                }
            } else if (kd_rem >= BK) {
#pragma unroll
                for (int s = 0; s < BK / 4; ++s) {
                    const uint8_t* so = sbase + (s >> 1) * 1024 + (s & 1) * 128;
                    double a[MI], b[NI];
#pragma unroll
                    for (int i = 0; i < MI; ++i)
                        a[i] = *reinterpret_cast<const double*>(so + (off_a(i) ^ ((uint32_t)(s & 1) << 4)));
#pragma unroll
                    for (int j = 0; j < NI; ++j)
                        b[j] = *reinterpret_cast<const double*>(so + (off_b(j) ^ ((uint32_t)(s & 1) << 4)));
#pragma unroll
                    for (int i = 0; i < MI; ++i)
#pragma unroll
                        for (int j = 0; j < NI; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
            } else {
                // last slab of the contraction: rows >= kd_rem are not part of it
#pragma unroll 1
                for (int s = 0; s < BK / 4; ++s) {
                    const int row = 8 * (s >> 1) + (s & 1) + 2 * lk;
                    const bool ok = row < kd_rem;
                    const uint8_t* so = sbase + (s >> 1) * 1024 + (s & 1) * 128;
                    double a[MI], b[NI];
#pragma unroll
                    for (int i = 0; i < MI; ++i) {
                        const double v = *reinterpret_cast<const double*>(so + (off_a(i) ^ ((uint32_t)(s & 1) << 4)));
                        a[i] = ok ? v : 0.0;
                    }
#pragma unroll
                    for (int j = 0; j < NI; ++j) {
                        const double v = *reinterpret_cast<const double*>(so + (off_b(j) ^ ((uint32_t)(s & 1) << 4)));
                        b[j] = ok ? v : 0.0;
                    }
#pragma unroll
                    for (int i = 0; i < MI; ++i)
#pragma unroll
                        for (int j = 0; j < NI; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_bar(stage));  // this warp is done with the stage
        }

        // ---- epilogue (as gemm_f64_kernel; the consumer warps synchronise on a named barrier) ----
        double* __restrict__ C = pr.C;
        const bool whole = (sg.kt0 == 0) && (sg.kt1 == sg.KT);
        const bool first_writer = (sg.kt1 == sg.KT);
        int* flag = batch.flags + pr.flag_begin + tile_lin;
        if (!whole && !first_writer) {
            const int tile_last_unit = sg.unit_begin + tile_lin * sg.KT + sg.KT - 1;
            const int after = (tile_last_unit - rem0) / upc - (int)blockIdx.x;
            if (tid == 0) {
                while (atomicAdd(flag, 0) < after) __nanosleep(64);
                __threadfence();
            }
            asm volatile("bar.sync 1, %0;\n" ::"r"(NCW * 32) : "memory");
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
            asm volatile("bar.sync 1, %0;\n" ::"r"(NCW * 32) : "memory");
            if (tid == 0) atomicAdd(flag, 1);
        }
    }
}

// ---- layout probe (ground truth for the swizzle / gather4 / out-of-bounds behaviour) -----------
// Loads one [BK=16][16] box with the tiled map at (col0, row0) and one 4-row gather at (col0,
// rows r[0..3]) and dumps the raw shared-memory images: out[0..255] tiled, out[256..319] gather.
__global__ void tma_probe_kernel(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapG,
                                 int col0, int row0, int4 rows, double* __restrict__ out) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar = base + 4096;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    for (int i = threadIdx.x; i < 320; i += blockDim.x) {
        const double nan_mark = -12345.0;
        asm volatile("st.shared.f64 [%0], %1;\n" ::"r"(base + 8u * (uint32_t)i), "d"(nan_mark));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // order the generic-proxy fills above before the async-proxy writes
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        mbar_arrive_expect_tx(bar, 16 * 128 + 4 * 128);
        tma_load_2d(base, &mapT, col0, row0, bar);
        tma_gather4(base + 2048, &mapG, col0, rows.x, rows.y, rows.z, rows.w, bar);
    }
    mbar_wait(bar, 0);
    for (int i = threadIdx.x; i < 320; i += blockDim.x) {
        double v;
        asm volatile("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(base + 8u * (uint32_t)i));
        out[i] = v;
    }
}

}  // namespace slm
