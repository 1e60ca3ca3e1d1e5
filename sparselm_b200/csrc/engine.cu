// sparselm_b200 engine: CUDA kernels (sm_100a) + C ABI (include/sparselm_b200.h).
//
// Kernel inventory (SURVEY.md section 2.2):
//   K1  gram build      gemm_f64_kernel<..., SYM>      (gemm_f64.cuh)   FP64 tensor
//   K2  centering       gram_center_kernel                             HBM
//   K3  overlap gather  gram_gather_kernel                             HBM
//   K4  lipschitz       gemm apply (N=8) + power_norm_kernel           HBM (N=8)
//   K5  gram apply      gemm_f64_kernel<...>                           FP64 tensor
//   K6  prox epilogue   prox_kernel  (momentum, soft-threshold, group shrink, ridge)
//   K7  gap + mask      gap_kernel   (duality gap, per-column convergence flag)
//   K8  reweighting     adaptive_kernel
//   K9  fold back       fold_back_kernel
//   K10 scoring         gemm_f64_kernel<A_MMAJOR> + score_kernel
//   K10b statistics     stat_residual/final/median_kernel (max, percentage sum, median of |r|)
//   K11 selection       support_colmax_kernel + support_count_kernel (stability selection counts)
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/sparselm_b200.h"
#include "gemm_f64.cuh"
#include "gemm_f64_tma.cuh"
#include "solver_kernels.cuh"
#include "whiten_kernels.cuh"
#include "cg_kernels.cuh"
#include "coop_kernels.cuh"
#include "newton_kernels.cuh"
#include "select_kernels.cuh"

using namespace slm;

// ------------------------------------------------------------------------- //
// context
// ------------------------------------------------------------------------- //
enum { FAM_GRAM = 0, FAM_APPLY = 1, FAM_PROX = 2, FAM_GAP = 3, FAM_SCORE = 4, FAM_LIPS = 5, FAM_COUNT = 6 };

struct Family {
    std::vector<cudaEvent_t> ev;  // begin/end pairs not yet accumulated
    std::vector<cudaEvent_t> pool;
    double ms = 0.0;
    double flops = 0.0;
    int64_t n = 0;
};

constexpr int kMaxScount = 4096;
constexpr int kMaxDevices = 64;  // function attributes are per device: launchers keep their one-time set-up per device

struct slm_ctx {
    int device = 0;
    int sm_count = 148;
    std::string err;
    int64_t launches = 0;
    int64_t tma_launches = 0;
    bool timing = false;
    bool newton_smem_set = false;  // the Newton kernels' dynamic shared-memory limits are raised on this device
    Family fam[FAM_COUNT];
    int* d_counter = nullptr;
    int* h_counter = nullptr;
    int* d_flags = nullptr;      // stream-K per-tile flags
    int n_flags_cap = 0;
    unsigned long long* d_stat = nullptr;  // executed contraction length of the row-sparse applies
    unsigned long long* h_stat = nullptr;
    unsigned long long* d_ratio = nullptr;  // worst gap / tolerance ratio of a convergence check
    unsigned long long* h_ratio = nullptr;
    int* h_scount = nullptr;         // pinned copy of the support-list lengths (chunk-width choice)
    double* h_scal = nullptr;        // pinned scalars of the conjugate-gradient loop
    unsigned long long* d_colmax = nullptr;  // [F][ldz] column maxima of slm_support_counts (grown on demand)
    size_t colmax_cap = 0;
    double apply_exec_flops = 0.0;   // flops the row-sparse applies executed (useful, unpadded)
    double apply_dense_flops = 0.0;  // 2 p^2 K_active of the same applies
    bool coop = true;                // SLM_COOP=0: never use the cooperative few-column iterations
    bool trace = false;              // SLM_TRACE=1: one stderr line per convergence check
    int coop_max_smem = 0;           // opt-in shared memory per block of the device
    int max_cluster = 16;            // largest cluster of the cluster kernel (8 where non-portable sizes are refused)
    int force_sparse_shape = -1;     // SLM_FORCE_SPARSE_SHAPE
    int force_apply_shape = -1;  // tuning/testing hook (SLM_FORCE_APPLY_SHAPE)
    int force_syrk_shape = -1;   // tuning/testing hook (SLM_FORCE_SYRK_SHAPE)
    // TMA-fed GEMM kernels (gemm_f64_tma.cuh): bit 0 Gram build, bit 1 dense apply, bit 2 row-sparse
    // apply (SLM_TMA / slm_set_option "tma"); encode = cuTensorMapEncodeTiled resolved at run time
    bool fused_prox = true;          // SLM_FUSED_PROX=0: the two-kernel iteration (prox_main + prox_momentum on the extrapolated point)
    int tma_mask = 7 + 8;  // + bit 3: wide bands for the gather kernels, bit 4: for the tiled kernels
    void* encode = nullptr;
};

static int fail(slm_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return code;
}
#define CUDA_OK(call)                                                                      \
    do {                                                                                   \
        cudaError_t e__ = (call);                                                          \
        if (e__ != cudaSuccess)                                                            \
            return fail(ctx, 100 + (int)e__,                                               \
                        std::string(#call) + ": " + cudaGetErrorString(e__));              \
    } while (0)
#define LAUNCH_OK(name)                                                                    \
    do {                                                                                   \
        cudaError_t e__ = cudaGetLastError();                                              \
        if (e__ != cudaSuccess)                                                            \
            return fail(ctx, 100 + (int)e__, std::string(name) + ": " + cudaGetErrorString(e__)); \
        ctx->launches++;                                                                   \
    } while (0)

struct FamTimer {  // RAII event pair around a launch when timing is on
    slm_ctx* ctx;
    int fam;
    cudaStream_t s;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    FamTimer(slm_ctx* c, int f, cudaStream_t st, double flops) : ctx(c), fam(f), s(st) {
        Family& F = ctx->fam[fam];
        F.flops += flops;
        F.n += 1;
        if (!ctx->timing) return;
        auto get = [&]() {
            cudaEvent_t e;
            if (!F.pool.empty()) {
                e = F.pool.back();
                F.pool.pop_back();
            } else {
                cudaEventCreate(&e);
            }
            return e;
        };
        e0 = get();
        e1 = get();
        cudaEventRecord(e0, s);
    }
    ~FamTimer() {
        if (!e0) return;
        cudaEventRecord(e1, s);
        ctx->fam[fam].ev.push_back(e0);
        ctx->fam[fam].ev.push_back(e1);
    }
};

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// ------------------------------------------------------------------------- //
// GEMM dispatch
// ------------------------------------------------------------------------- //
constexpr int kBK = 16;
constexpr int kStages = 4;

struct Shape {
    int bm, bn;
    int minb;   // CTAs per SM the kernel is built for
    double eff; // measured fraction of the per-SM DMMA peak this warp layout reaches
};

static void fill_units(GemmBatch& b, int bm, int bn, bool sym, int max_ctas, int bk = kBK, bool waves = true) {
    long long u = 0;
    int nflags = 0;
    for (int i = 0; i < b.n_problems; ++i) {
        GemmProblem& pr = b.pr[i];
        if (pr.qlim <= 0) pr.qlim = (int)pr.ldq;
        pr.tiles_m = (pr.M + bm - 1) / bm;
        pr.tiles_n = (pr.N + bn - 1) / bn;
        pr.kt = std::max(1, (pr.Kd + bk - 1) / bk);
        if (pr.N <= 0 || pr.M <= 0 || pr.Kd <= 0) pr.tiles_m = pr.tiles_n = 0;
        pr.n_tiles = sym ? pr.tiles_n * (pr.tiles_n + 1) / 2 : pr.tiles_m * pr.tiles_n;
        pr.unit_begin = (int)u;
        pr.flag_begin = nflags;
        pr.tile_begin = nflags;
        nflags += pr.n_tiles;
        u += (long long)pr.n_tiles * pr.kt;
    }
    b.total_units = (int)u;
    b.n_flags = nflags;
    // persistent grid: every CTA is resident.  Whole waves of tiles are data-parallel (one tile
    // per CTA, the CTAs of a wave sweep k together and share operand panels in L2); the units of
    // the partial last wave are cut into equal ranges => the SMs still finish together
    long long n_cta = std::min<long long>(max_ctas, std::max<long long>(1, u));
    b.full_waves = 0;
    b.rem_unit_begin = 0;
    if (waves && nflags >= n_cta && n_cta == max_ctas) {
        b.full_waves = (int)(nflags / n_cta);
        const int t0 = b.full_waves * (int)n_cta;  // first tile of the stream-K remainder
        long long u0 = u;
        for (int i = 0; i < b.n_problems; ++i) {
            const GemmProblem& pr = b.pr[i];
            if (t0 >= pr.tile_begin && t0 < pr.tile_begin + pr.n_tiles)
                u0 = pr.unit_begin + (long long)(t0 - pr.tile_begin) * pr.kt;
        }
        b.rem_unit_begin = (int)u0;
    }
    const long long rem = u - b.rem_unit_begin;
    b.units_per_cta = (int)std::max<long long>(1, (rem + n_cta - 1) / n_cta);
}

template <int WM, int WN, int MI, int NI, bool AM, bool SYM, int MINB, bool KSP = false, int BK = kBK,
          int STAGES = kStages, bool AG = false>
static cudaError_t launch_gemm_t(slm_ctx* ctx, GemmBatch& b, cudaStream_t s) {
    using Cfg = GemmCfg<WM, WN, MI, NI, BK, STAGES, AM>;
    auto kern = gemm_f64_kernel<WM, WN, MI, NI, BK, STAGES, AM, SYM, MINB, KSP, AG>;
    // resident CTAs per SM (the spin-wait fix-up needs co-residency); the shared-memory limit is raised per device
    static int occupancy_of[kMaxDevices] = {};
    if (ctx->device >= kMaxDevices) return cudaErrorInvalidDevice;
    int& occupancy = occupancy_of[ctx->device];
    if (occupancy == 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)Cfg::SMEM);
        if (e != cudaSuccess) return e;
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, Cfg::NT, Cfg::SMEM);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occupancy = std::min(occ, MINB);
    }
    fill_units(b, Cfg::BM, Cfg::BN, SYM, ctx->sm_count * occupancy, BK);
    if (b.total_units <= 0) return cudaSuccess;
    if (b.n_flags > ctx->n_flags_cap) return cudaErrorInvalidValue;
    b.flags = ctx->d_flags;
    int grid = b.full_waves > 0 ? ctx->sm_count * occupancy : (b.total_units + b.units_per_cta - 1) / b.units_per_cta;
    // row-sparse apply: the k extents live on the device, the CTAs partition the units themselves
    if (KSP && !SYM) grid = (int)std::min<long long>((long long)ctx->sm_count * occupancy, b.total_units);
    cudaError_t e = cudaMemsetAsync(b.flags, 0, sizeof(int) * (size_t)b.n_flags, s);
    if (e != cudaSuccess) return e;
    kern<<<grid, Cfg::NT, Cfg::SMEM, s>>>(b);
    return cudaGetLastError();
}


// ---- TMA-fed variants ------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D map over a row-major [rows][ld] FP64 matrix, boxes of [box_rows][16 doubles], 128-byte swizzle,
// out-of-bounds elements read as zero
static bool make_map(slm_ctx* ctx, CUtensorMap* map, const double* base, long long rows, long long ld, int box_rows,
                     int box_cols = kTmaBoxCols, bool swizzle = true) {
    if (!ctx->encode || !base || rows <= 0 || ld <= 0 || (ld & 1) || ((uintptr_t)base & 15)) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(double)};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = ((EncodeTiledFn)ctx->encode)(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, gdim, gstr, box, estr,
                                              CU_TENSOR_MAP_INTERLEAVE_NONE,
                                              swizzle ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// can this batch run on the TMA kernels?  Fills prow0 / pcol0 / qrow0 / qcol0 of every problem.
static bool tma_prepare(slm_ctx* ctx, GemmBatch& b, int family_bit) {
    if (!(ctx->tma_mask & family_bit) || !ctx->encode || !b.baseP || !b.baseQ) return false;
    for (int i = 0; i < b.n_problems; ++i) {
        GemmProblem& pr = b.pr[i];
        if (pr.ldp != b.pr[0].ldp || pr.ldq != b.pr[0].ldq) return false;
        const long long dp = pr.P - b.baseP, dq = pr.Q - b.baseQ;
        if (dp < 0 || dq < 0 || ((dp % pr.ldp) & 1) || ((dq % pr.ldq) & 1)) return false;  // box starts are 16-byte aligned
        pr.prow0 = (int)(dp / pr.ldp);
        pr.pcol0 = (int)(dp % pr.ldp);
        pr.qrow0 = (int)(dq / pr.ldq);
        pr.qcol0 = (int)(dq % pr.ldq);
        if ((long long)pr.prow0 + pr.Kd > (1LL << 30) || (long long)pr.qrow0 + pr.Kd > (1LL << 30)) return false;
    }
    return true;
}

template <int WM, int WN, int MI, int NI, bool SYM, int MINB, bool KSP, int BK, int STAGES, bool WIDE>
static cudaError_t launch_gemm_tma_w(slm_ctx* ctx, GemmBatch& b, cudaStream_t s) {
    using Cfg = TmaCfg<WM, WN, MI, NI, BK, STAGES, WIDE>;
    auto kern = gemm_f64_tma_kernel<WM, WN, MI, NI, BK, STAGES, SYM, MINB, KSP, WIDE>;
    static int occupancy_of[kMaxDevices] = {};  // per device, like the shared-memory limit it is measured with
    if (ctx->device >= kMaxDevices) return cudaErrorInvalidDevice;
    int& occupancy = occupancy_of[ctx->device];
    if (occupancy == 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
        if (e != cudaSuccess) return e;
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, Cfg::NT, Cfg::SMEM);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occupancy = std::min(occ, MINB);
    }
    fill_units(b, Cfg::BM, Cfg::BN, SYM, ctx->sm_count * occupancy, BK);
    if (b.total_units <= 0) return cudaSuccess;
    if (b.n_flags > ctx->n_flags_cap) return cudaErrorInvalidValue;
    b.flags = ctx->d_flags;
    CUtensorMap mp, mq;
    const int box_rows = KSP ? 1 : BK;
    if (!make_map(ctx, &mp, b.baseP, b.rowsP, b.pr[0].ldp, box_rows, Cfg::A_COLS, !WIDE) ||
        !make_map(ctx, &mq, b.baseQ, b.rowsQ, b.pr[0].ldq, box_rows, Cfg::B_COLS, !WIDE))
        return cudaErrorInvalidValue;
    int grid = b.full_waves > 0 ? ctx->sm_count * occupancy : (b.total_units + b.units_per_cta - 1) / b.units_per_cta;
    if (KSP && !SYM) grid = (int)std::min<long long>((long long)ctx->sm_count * occupancy, b.total_units);
    cudaError_t e = cudaMemsetAsync(b.flags, 0, sizeof(int) * (size_t)b.n_flags, s);
    if (e != cudaSuccess) return e;
    kern<<<grid, Cfg::NT, Cfg::SMEM, s>>>(b, mp, mq);
    ctx->tma_launches++;
    return cudaGetLastError();
}

// layout choice (tma_mask bit 3 = wide bands for the gather kernels, bit 4 = wide bands for the tiled ones)
template <int WM, int WN, int MI, int NI, bool SYM, int MINB, bool KSP, int BK, int STAGES>
static cudaError_t launch_gemm_tma_t(slm_ctx* ctx, GemmBatch& b, cudaStream_t s) {
    const bool wide = (ctx->tma_mask & (KSP ? 8 : 16)) != 0;
    if (wide) return launch_gemm_tma_w<WM, WN, MI, NI, SYM, MINB, KSP, BK, STAGES, true>(ctx, b, s);
    return launch_gemm_tma_w<WM, WN, MI, NI, SYM, MINB, KSP, BK, STAGES, false>(ctx, b, s);
}

// K-major (apply) menu.  X(id, WM, WN, MI, NI, MINB, eff): tile = (WM*MI*8) x (WN*NI*8);
// eff = measured fraction of the per-SM DMMA peak of that warp layout (profiles/).
#define SLM_APPLY_SHAPES(X)        \
    X(0, 2, 4, 8, 4, 1, 0.76)      \
    X(1, 8, 1, 2, 13, 1, 0.72)     \
    X(2, 16, 1, 1, 13, 1, 0.776)   \
    X(3, 8, 1, 2, 7, 2, 0.765)     \
    X(4, 4, 4, 4, 4, 1, 0.80)      \
    X(5, 4, 2, 4, 4, 2, 0.78)      \
    X(6, 8, 1, 1, 13, 2, 0.74)     \
    X(7, 8, 1, 2, 4, 2, 0.84)      \
    X(8, 8, 1, 2, 2, 2, 0.70)      \
    X(9, 8, 1, 2, 1, 2, 0.55)      \
    X(10, 8, 1, 2, 3, 2, 0.78)     \
    X(11, 8, 1, 2, 5, 2, 0.80)     \
    X(12, 8, 1, 2, 6, 2, 0.79)     \
    X(13, 16, 1, 1, 9, 1, 0.775)   \
    X(14, 16, 1, 1, 10, 1, 0.775)  \
    X(15, 16, 1, 1, 11, 1, 0.775)  \
    X(16, 16, 1, 1, 12, 1, 0.775)

static const Shape kApplyShapes[] = {
#define X(id, wm, wn, mi, ni, minb, eff) {wm * mi * 8, wn * ni * 8, minb, eff},
    SLM_APPLY_SHAPES(X)
#undef X
};
constexpr int kNumApplyShapes = sizeof(kApplyShapes) / sizeof(Shape);

static cudaError_t launch_apply_shape(slm_ctx* ctx, int id, GemmBatch& b, cudaStream_t s) {
    if (tma_prepare(ctx, b, 2)) {
        switch (id) {
#define X(id_, wm, wn, mi, ni, minb, eff) \
    case id_: return launch_gemm_tma_t<wm, wn, mi, ni, false, minb, false, kBK, kStages>(ctx, b, s);
            SLM_APPLY_SHAPES(X)
#undef X
        }
    }
    switch (id) {
#define X(id_, wm, wn, mi, ni, minb, eff) \
    case id_: return launch_gemm_t<wm, wn, mi, ni, false, false, minb>(ctx, b, s);
        SLM_APPLY_SHAPES(X)
#undef X
    }
    return cudaErrorInvalidValue;
}
// row-sparse apply menu (one tile column per support chunk): id, WM, WN, MI, NI, MINB, eff
// narrow tiles run 3 CTAs (24 warps) per SM with a 3-stage pipeline: measured 6.6 % faster than
// 2 CTAs x 4 stages on the mid-solve scenario of tools/apply_probe.py (more warps hide the
// gather latency; 80 registers, no spills)
// eff: measured with the TMA wide-band kernels (tools/gemm_probe.py, profiles/r02c_gemm_probe.txt).  A tile
// re-reads its 128-column band of the support rows of G whatever its width: below ~40 columns the tile time
// is set by that L2 -> shared-memory traffic, not by the DMMA pipe, so the efficiency of narrow tiles
// falls in proportion to their width (a 16-column tile costs what a 32-column tile costs).
#define SLM_SPARSE_SHAPES(X)      \
    X(0, 8, 1, 2, 1, 3, 0.18)     \
    X(1, 8, 1, 2, 2, 3, 0.36)     \
    X(2, 8, 1, 2, 3, 3, 0.54)     \
    X(3, 8, 1, 2, 4, 3, 0.72)     \
    X(4, 8, 1, 2, 5, 3, 0.76)     \
    X(5, 8, 1, 2, 6, 3, 0.78)     \
    X(6, 8, 1, 2, 7, 2, 0.78)     \
    X(7, 4, 2, 4, 4, 2, 0.78)     \
    X(8, 16, 1, 1, 9, 1, 0.82)    \
    X(9, 16, 1, 1, 11, 1, 0.86)   \
    X(10, 16, 1, 1, 13, 1, 0.90)  \
    X(11, 2, 4, 8, 4, 1, 0.76)    \
    X(12, 8, 1, 2, 13, 1, 0.88)   \
    X(13, 8, 1, 2, 8, 2, 0.78)
static const Shape kSparseShapes[] = {
#define X(id, wm, wn, mi, ni, minb, eff) {wm * mi * 8, wn * ni * 8, minb, eff},
    SLM_SPARSE_SHAPES(X)
#undef X
};
constexpr int kNumSparseShapes = sizeof(kSparseShapes) / sizeof(Shape);
static cudaError_t launch_sparse_shape(slm_ctx* ctx, int id, GemmBatch& b, cudaStream_t s) {
    // tiles of <= 16 columns run a few microseconds per launch: the cp.async kernel starts faster there
    // (no barrier ring / register re-allocation / descriptor fetch), measured in tools/gemm_probe.py
    if (kSparseShapes[id].bn > 16 && tma_prepare(ctx, b, 4)) {
        switch (id) {
#define X(id_, wm, wn, mi, ni, minb, eff) \
    case id_: return launch_gemm_tma_t<wm, wn, mi, ni, false, minb, true, kBK, (minb >= 3 ? 3 : kStages)>(ctx, b, s);
            SLM_SPARSE_SHAPES(X)
#undef X
        }
    }
    switch (id) {
#define X(id_, wm, wn, mi, ni, minb, eff) \
    case id_: return launch_gemm_t<wm, wn, mi, ni, false, false, minb, true, kBK, (minb >= 3 ? 3 : kStages)>(ctx, b, s);
        SLM_SPARSE_SHAPES(X)
#undef X
    }
    return cudaErrorInvalidValue;
}
// M-major (scoring) menu
static const Shape kScoreShapes[] = {{128, 128, 1, 0.84}, {128, 64, 2, 0.85}, {128, 32, 2, 0.8}, {128, 16, 2, 0.7}, {128, 8, 2, 0.6}};
constexpr int kNumScoreShapes = sizeof(kScoreShapes) / sizeof(Shape);
static cudaError_t launch_score_shape(slm_ctx* ctx, int id, GemmBatch& b, cudaStream_t s) {
    switch (id) {
        case 0: return launch_gemm_t<2, 4, 8, 4, true, false, 1>(ctx, b, s);
        case 1: return launch_gemm_t<4, 2, 4, 4, true, false, 2>(ctx, b, s);
        case 2: return launch_gemm_t<8, 1, 2, 4, true, false, 2>(ctx, b, s);
        case 3: return launch_gemm_t<8, 1, 2, 2, true, false, 2>(ctx, b, s);
        case 4: return launch_gemm_t<8, 1, 2, 1, true, false, 2>(ctx, b, s);
    }
    return cudaErrorInvalidValue;
}
// symmetric (Gram build) menu: 128x128 tiles.  Measured at the C3 shape (tools/syrk_probe.py):
// a 32-deep k-slab (half as many CTA-wide barriers per flop) with 3 stages beats 16-deep x 4
// stages by 9 % (11.25 vs 12.26 ms); more warps or other warp tiles change little.
static cudaError_t launch_syrk_shape(slm_ctx* ctx, int id, GemmBatch& b, cudaStream_t s) {
    if (id <= 1 && tma_prepare(ctx, b, 1)) {
        if (id == 0) return launch_gemm_tma_t<2, 4, 8, 4, true, 1, false, 32, 3>(ctx, b, s);
        return launch_gemm_tma_t<4, 4, 4, 4, true, 1, false, 32, 3>(ctx, b, s);
    }
    switch (id) {
        case 0: return launch_gemm_t<2, 4, 8, 4, false, true, 1, false, 32, 3>(ctx, b, s);
        case 1: return launch_gemm_t<4, 4, 4, 4, false, true, 1, false, 32, 3>(ctx, b, s);
        case 2: return launch_gemm_t<2, 4, 8, 4, false, true, 1>(ctx, b, s);
        case 3: return launch_gemm_t<4, 4, 4, 4, false, true, 1>(ctx, b, s);
    }
    return cudaErrorInvalidValue;
}
constexpr int kNumSyrkShapes = 4;
// gathered Gram (slm_gram_rows_update): the 128 x 128, 32-deep-slab shape of the Gram build, its rows
// gathered by the TMA unit (tile::gather4) or by the cp.async copies
static cudaError_t launch_syrk_rows(slm_ctx* ctx, GemmBatch& b, cudaStream_t s) {
    if (tma_prepare(ctx, b, 1)) return launch_gemm_tma_t<2, 4, 8, 4, true, 1, true, 32, 3>(ctx, b, s);
    return launch_gemm_t<2, 4, 8, 4, false, true, 1, true, 32, 3>(ctx, b, s);
}
// scoring GEMM over gathered rows of Xa (slm_cv_score_rows): the scoring menu, A rows gathered
static cudaError_t launch_score_rows_shape(slm_ctx* ctx, int id, GemmBatch& b, cudaStream_t s) {
    switch (id) {
        case 0: return launch_gemm_t<2, 4, 8, 4, true, false, 1, false, kBK, kStages, true>(ctx, b, s);
        case 1: return launch_gemm_t<4, 2, 4, 4, true, false, 2, false, kBK, kStages, true>(ctx, b, s);
        case 2: return launch_gemm_t<8, 1, 2, 4, true, false, 2, false, kBK, kStages, true>(ctx, b, s);
        case 3: return launch_gemm_t<8, 1, 2, 2, true, false, 2, false, kBK, kStages, true>(ctx, b, s);
        case 4: return launch_gemm_t<8, 1, 2, 1, true, false, 2, false, kBK, kStages, true>(ctx, b, s);
    }
    return cudaErrorInvalidValue;
}

struct ProblemDims {
    int M, N;
};
// cost model: the kernel is DMMA-bound and stream-K balances the SMs, so time is
// (padded tile work) / (efficiency of the warp layout).
static int pick_shape(const Shape* shapes, int n_shapes, const ProblemDims* pd, int np, int sms) {
    (void)sms;
    int best = 0;
    double best_cost = 1e300;
    for (int s = 0; s < n_shapes; ++s) {
        double work = 0.0;
        for (int i = 0; i < np; ++i) {
            if (pd[i].N <= 0) continue;
            work += (double)((pd[i].M + shapes[s].bm - 1) / shapes[s].bm) *
                    ((pd[i].N + shapes[s].bn - 1) / shapes[s].bn) * shapes[s].bm * shapes[s].bn;
        }
        double cost = work / shapes[s].eff;
        if (cost < best_cost) {
            best_cost = cost;
            best = s;
        }
    }
    return best;
}

// batched apply: GZ_f = G_f Z_f for f < F, with N_f = round_up(K_f, 8)
static int apply_batched(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int F,
                         const int32_t* K, const double* Z, int64_t ldz, double* GZ, cudaStream_t s,
                         double algo_flops = -1.0, int family = FAM_APPLY) {
    for (int f0 = 0; f0 < F; f0 += kMaxGemmProblems) {
        int nf = std::min(F - f0, (int)kMaxGemmProblems);
        GemmBatch b;
        memset(&b, 0, sizeof(b));
        ProblemDims pd[kMaxGemmProblems];
        double flops = 0.0;
        b.n_problems = nf;
        if (g_stride % pa == 0) {  // the Grams are row blocks of one [rows][pa] matrix: TMA-addressable
            b.baseP = G;
            b.rowsP = (int64_t)(F - 1) * (g_stride / pa) + pa;
            b.baseQ = Z;
            b.rowsQ = (int64_t)F * p;
        }
        for (int i = 0; i < nf; ++i) {
            int f = f0 + i;
            GemmProblem& pr = b.pr[i];
            pr.P = G + (int64_t)f * g_stride;
            pr.Q = Z + (int64_t)f * p * ldz;
            pr.C = GZ + (int64_t)f * p * ldz;
            pr.ldp = pa;
            pr.ldq = ldz;
            pr.ldc = ldz;
            pr.M = (int)p;
            pr.N = (int)std::min<int64_t>(round_up(K[f], 8), ldz);
            pr.Kd = (int)p;
            pd[i] = {pr.M, pr.N};
            flops += 2.0 * (double)p * (double)p * (double)K[f];
        }
        int sid = pick_shape(kApplyShapes, kNumApplyShapes, pd, nf, ctx->sm_count);
        if (ctx->force_apply_shape >= 0 && ctx->force_apply_shape < kNumApplyShapes) sid = ctx->force_apply_shape;
        FamTimer tm(ctx, family, s, algo_flops >= 0 ? algo_flops : flops);
        cudaError_t e = launch_apply_shape(ctx, sid, b, s);
        if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("gram apply: ") + cudaGetErrorString(e));
        ctx->launches++;
    }
    return 0;
}

// row-sparse batched apply: GZ_f = G_f Z_f using only the rows of Z_f that hold a non-zero
// in the column chunk (chunks of chunk_w columns; lists made by support_list_kernel from
// the zflag bytes).  ncc = chunk slots per fold in sidx / scount.
static int apply_rowsparse(slm_ctx* ctx, const SolveDev& sp, const int32_t* K, const double* Z, double* GZ,
                           int chunk_w, int ncc, int* sidx, int* scount, cudaStream_t s, double algo_flops) {
    const int F = sp.F;
    const int64_t p = sp.p, ldz = sp.ldz;
    support_list_kernel<<<dim3((unsigned)ncc, (unsigned)F), 1024, 0, s>>>(sp, chunk_w / SC, ncc, sidx, scount,
                                                                          ctx->d_stat);
    LAUNCH_OK("support_list_kernel");
    GemmBatch b;
    ProblemDims pd[kMaxGemmProblems];
    int np = 0;
    double dense = 0.0;
    bool first = true;
    auto flush = [&]() -> int {
        if (np == 0) return 0;
        b.n_problems = np;
        if (sp.g_stride % sp.pa == 0) {
            b.baseP = sp.G;
            b.rowsP = (int64_t)(F - 1) * (sp.g_stride / sp.pa) + sp.pa;
            b.baseQ = Z;
            b.rowsQ = (int64_t)F * p;
        }
        int sid = pick_shape(kSparseShapes, kNumSparseShapes, pd, np, ctx->sm_count);
        if (ctx->force_sparse_shape >= 0 && ctx->force_sparse_shape < 14) sid = ctx->force_sparse_shape;
        FamTimer tm(ctx, FAM_APPLY, s, first ? std::max(algo_flops, 0.0) : 0.0);
        first = false;
        cudaError_t e = launch_sparse_shape(ctx, sid, b, s);
        if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("row-sparse apply: ") + cudaGetErrorString(e));
        ctx->launches++;
        np = 0;
        return 0;
    };
    memset(&b, 0, sizeof(b));
    for (int f = 0; f < F; ++f) {
        const int Kp = (int)std::min<int64_t>(round_up(K[f], 8), ldz);
        dense += 2.0 * (double)p * (double)p * (double)K[f];
        for (int cc = 0; cc * chunk_w < Kp; ++cc) {
            if (np == kMaxGemmProblems) {
                int rc = flush();
                if (rc) return rc;
                memset(&b, 0, sizeof(b));
            }
            GemmProblem& pr = b.pr[np];
            const int64_t off = (int64_t)f * p * ldz + (int64_t)cc * chunk_w;
            pr.P = sp.G + (int64_t)f * sp.g_stride;
            pr.Q = Z + off;
            pr.C = GZ + off;
            pr.kidx = sidx + ((int64_t)f * ncc + cc) * p;
            pr.kcount = scount + f * ncc + cc;
            pr.ldp = sp.pa;
            pr.ldq = pr.ldc = ldz;
            pr.qlim = (int)(ldz - (int64_t)cc * chunk_w);
            pr.M = (int)p;
            pr.N = std::min(chunk_w, Kp - cc * chunk_w);
            pr.Kd = (int)p;
            pd[np] = {pr.M, pr.N};
            ++np;
        }
    }
    ctx->apply_dense_flops += dense;
    return flush();
}

// ------------------------------------------------------------------------- //
// small kernels: packing, complement, centering, gather
// ------------------------------------------------------------------------- //
__global__ void pack_design_kernel(const double* __restrict__ X, long long ldx,
                                   const double* __restrict__ y, const double* __restrict__ sw,
                                   const int* __restrict__ col_perm,
                                   const long long* __restrict__ row_perm, long long n, int p,
                                   double* __restrict__ Xa, long long lda) {
    long long r = blockIdx.y;
    long long src_r = row_perm ? row_perm[r] : r;
    double s = sw ? sqrt(sw[src_r]) : 1.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < lda; j += gridDim.x * blockDim.x) {
        double v;
        if (j < p) {
            int sj = col_perm ? col_perm[j] : j;
            v = s * X[src_r * ldx + sj];
        } else if (j == p) {
            v = s * y[src_r];
        } else if (j == p + 1) {
            v = s;
        } else {
            v = 0.0;
        }
        Xa[r * lda + j] = v;
    }
}

__global__ void gram_complement_kernel(double* __restrict__ Gblk, int nb, long long stride,
                                       double* __restrict__ Gtot) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= stride) return;
    double vals[SLM_MAX_FOLDS];
    double tot = 0.0;
    for (int f = 0; f < nb; ++f) {
        vals[f] = Gblk[(long long)f * stride + i];
        tot += vals[f];
    }
    Gtot[i] = tot;
    for (int f = 0; f < nb; ++f) {
        // sum of the other blocks in a fixed order (no subtraction => no cancellation)
        double acc = 0.0;
        for (int g = 0; g < nb; ++g)
            if (g != f) acc += vals[g];
        Gblk[(long long)f * stride + i] = acc;
    }
}

// symmetric Gram <-> packed upper triangle (row i holds columns i..pa-1): the row-sharded
// build only sends the upper triangles through the all-reduce
__device__ __forceinline__ long long tri_off(long long i, long long pa) { return i * pa - i * (i - 1) / 2; }
__global__ void tri_pack_kernel(const double* __restrict__ G, long long g_stride, long long pa,
                                double* __restrict__ buf, long long b_stride) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = blockIdx.y;
    if (j >= pa || j < i) return;
    buf[(long long)blockIdx.z * b_stride + tri_off(i, pa) + (j - i)] = G[(long long)blockIdx.z * g_stride + i * pa + j];
}
__global__ void tri_unpack_kernel(const double* __restrict__ buf, long long b_stride, long long pa,
                                  double* __restrict__ G, long long g_stride) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = blockIdx.y;
    if (j >= pa) return;
    const double* b = buf + (long long)blockIdx.z * b_stride;
    const double v = j >= i ? b[tri_off(i, pa) + (j - i)] : b[tri_off(j, pa) + (i - j)];
    G[(long long)blockIdx.z * g_stride + i * pa + j] = v;
}

// packed upper triangles of the F fold blocks -> the F training Grams (sum of the OTHER blocks, fixed
// order, no subtraction) and the total, full symmetric matrices: tri_unpack + gram_complement in one
// pass over the reduced buffer (the sharded build's tail: 1.1 GB of traffic instead of 2.4 GB at C3)
__global__ void tri_complement_kernel(const double* __restrict__ buf, long long b_stride, long long pa, int nb,
                                      double* __restrict__ G, long long g_stride) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long i = blockIdx.y;
    if (j >= pa || j < i) return;
    const long long t = tri_off(i, pa) + (j - i);
    double vals[SLM_MAX_FOLDS];
    double tot = 0.0;
    for (int f = 0; f < nb; ++f) {
        vals[f] = buf[(long long)f * b_stride + t];
        tot += vals[f];
    }
    for (int f = 0; f <= nb; ++f) {
        double acc = tot;
        if (f < nb) {
            acc = 0.0;
            for (int g = 0; g < nb; ++g)
                if (g != f) acc += vals[g];
        }
        double* Gf = G + (long long)f * g_stride;
        Gf[i * pa + j] = acc;
        if (j != i) Gf[j * pa + i] = acc;
    }
}

__global__ void gram_center_kernel(double* __restrict__ G, long long pa, int p) {
    // rows/cols 0..p (features and y); ones row p+1 kept intact
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j > p || i > p) return;
    const double* ones = G + (long long)(p + 1) * pa;
    double n = ones[p + 1];
    G[(long long)i * pa + j] -= ones[i] * ones[j] / n;
}

__global__ void gram_gather_kernel(const double* __restrict__ G, long long pa, int p,
                                   const int* __restrict__ idx, int pe, double* __restrict__ Ge,
                                   long long pae) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    int a = blockIdx.y;
    if (b >= pae) return;
    double v = 0.0;
    if (a < pe + 2 && b < pe + 2) {
        int ia = a < pe ? idx[a] : p + (a - pe);
        int ib = b < pe ? idx[b] : p + (b - pe);
        v = G[(long long)ia * pa + ib];
    }
    Ge[(long long)a * pae + b] = v;
}

// ------------------------------------------------------------------------- //
// solver kernels
// ------------------------------------------------------------------------- //
constexpr int CT = 4;          // grid columns per block (adaptive kernel)
constexpr int PT = 256;        // threads per block
constexpr int NGL = PT / CT;   // group lanes per block

template <typename T>
__device__ __forceinline__ T block_col_reduce_sum(T v, T (*red)[CT], int gl, int c) {
    red[gl][c] = v;
    __syncthreads();
#pragma unroll
    for (int s = NGL / 2; s > 0; s >>= 1) {
        if (gl < s) red[gl][c] += red[gl + s][c];
        __syncthreads();
    }
    T r = red[0][c];
    __syncthreads();
    return r;
}

__global__ void init_cols_kernel(double* theta, double* tmom, int* flag, int* colmap, int* status, int* n_iter,
                                 const int* skip, long long n, int ldz) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    theta[i] = theta[n + i] = 0.0;  // both parities
    tmom[i] = tmom[n + i] = 1.0;
    colmap[i] = (int)(i % ldz);
    if (skip && skip[i]) {
        flag[i] = 3;  // frozen by the caller; results of the earlier solve are kept
        return;
    }
    flag[i] = 0;
    if (status) status[i] = -1;
    if (n_iter) n_iter[i] = 0;
}

// K4 helper: V <- W/||W|| per column, tracks the largest Rayleigh quotient.
// One CTA per Gram, 8 columns x PN_LANES row lanes (a sharded rank holds one or two Grams, so
// the kernel is latency-bound: many lanes, independent loads).
constexpr int PN_LANES = 128;
__global__ void __launch_bounds__(8 * PN_LANES) power_norm_kernel(double* __restrict__ V, const double* __restrict__ W,
                                                                  int p, double* __restrict__ lam, int init) {
    const int f = blockIdx.x;
    const int c = threadIdx.x & 7, r = threadIdx.x >> 3;  // 8 columns x PN_LANES row lanes
    double* Vf = V + (long long)f * p * 8;
    const double* Wf = W + (long long)f * p * 8;
    __shared__ double red[3][PN_LANES][8];
    if (init) {
        for (int j = r; j < p; j += PN_LANES) {
            unsigned h = (unsigned)(j * 8 + c) * 2654435761u + 12345u * (unsigned)(f + 1);
            h ^= h >> 15;
            h *= 2246822519u;
            h ^= h >> 13;
            Vf[(long long)j * 8 + c] = ((double)(h & 0xffffff) / 8388608.0) - 1.0;
        }
        if (threadIdx.x == 0) lam[f] = 0.0;
        return;
    }
    double vw = 0.0, ww = 0.0, vv = 0.0;
    for (int j = r; j < p; j += PN_LANES) {
        double v = Vf[(long long)j * 8 + c], w = Wf[(long long)j * 8 + c];
        vw += v * w;
        ww += w * w;
        vv += v * v;
    }
    red[0][r][c] = vw;
    red[1][r][c] = ww;
    red[2][r][c] = vv;
    __syncthreads();
    for (int s = PN_LANES / 2; s > 0; s >>= 1) {
        if (r < s) {
            red[0][r][c] += red[0][r + s][c];
            red[1][r][c] += red[1][r + s][c];
            red[2][r][c] += red[2][r + s][c];
        }
        __syncthreads();
    }
    vw = red[0][0][c];
    ww = red[1][0][c];
    vv = red[2][0][c];
    if (threadIdx.x == 0) {
        double best = lam[f];
        for (int cc = 0; cc < 8; ++cc) {
            double q = red[2][0][cc] > 0.0 ? red[0][0][cc] / red[2][0][cc] : 0.0;
            best = fmax(best, q);
        }
        lam[f] = best;
    }
    const double inv = ww > 0.0 ? rsqrt(ww) : 0.0;
    for (int j = r; j < p; j += PN_LANES) Vf[(long long)j * 8 + c] = Wf[(long long)j * 8 + c] * inv;
}

// K8: adaptive reweighting.
__global__ void __launch_bounds__(PT) adaptive_kernel(const double* __restrict__ B, int p, long long ldz, int K,
                                                      int Gn, const int* __restrict__ gptr,
                                                      const double* __restrict__ gw,
                                                      const double* __restrict__ a1,
                                                      const double* __restrict__ a2,
                                                      const double* __restrict__ alpha, double eps,
                                                      double* __restrict__ W1, double* __restrict__ W2,
                                                      double* __restrict__ dnorm) {
    const int k0 = blockIdx.x * CT;
    const int c = threadIdx.x % CT, gl = threadIdx.x / CT;
    const int k = k0 + c;
    const bool colok = k < K;
    __shared__ double red[NGL][CT];
    double acc = 0.0;
    if (colok) {
        const double al = alpha[k];
        const double s1 = a1 ? a1[k] : 0.0;
        const double s2 = a2 ? a2[k] : 0.0;
        for (int g = gl; g < Gn; g += NGL) {
            const int ja = gptr ? gptr[g] : g;
            const int jb = gptr ? gptr[g + 1] : g + 1;
            double ss = 0.0;
            for (int j = ja; j < jb; ++j) {
                const double b = B[(long long)j * ldz + k];
                ss += b * b;
                if (W1) {
                    const double wn = s1 * (al / (fabs(b) + eps));
                    const double d = wn - W1[(long long)j * ldz + k];
                    acc += d * d;
                    W1[(long long)j * ldz + k] = wn;
                }
            }
            if (W2) {
                const double wn = (s2 * (gw ? gw[g] : 1.0)) * (al / (sqrt(ss) + eps));
                const double d = wn - W2[(long long)g * ldz + k];
                acc += d * d;
                W2[(long long)g * ldz + k] = wn;
            }
        }
    }
    acc = block_col_reduce_sum<double>(acc, red, gl, c);
    if (colok && gl == 0 && dnorm) dnorm[k] = sqrt(acc);
}

// K9
__global__ void fold_back_kernel(const double* __restrict__ Be, const int* __restrict__ inv_ptr,
                                 const int* __restrict__ inv_idx, int p, long long ldz, int K,
                                 double* __restrict__ coef) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    int j = blockIdx.y;
    if (k >= K || j >= p) return;
    double acc = 0.0;
    for (int t = inv_ptr[j]; t < inv_ptr[j + 1]; ++t) acc += Be[(long long)inv_idx[t] * ldz + k];
    coef[(long long)j * ldz + k] = acc;
}

// K10: residual reductions, two deterministic stages.
constexpr int SCORE_RB = 128;  // row blocks
// GATHER: row i of the problem is row ridx[i] of Xa (r0 unused), else row r0 + i
template <bool GATHER = false>
__global__ void __launch_bounds__(256) score_partial_kernel(const double* __restrict__ Xa, long long lda, int p,
                                                            long long r0, long long m,
                                                            const double* __restrict__ yhat, long long ldz,
                                                            int K, const double* __restrict__ icpt,
                                                            int rows_scaled, double* __restrict__ part,
                                                            const int* __restrict__ ridx = nullptr) {
    // block = 8 columns x 32 row lanes; grid = (ceil(K/8), SCORE_RB)
    const int c = threadIdx.x & 7, r = threadIdx.x >> 3;
    const int k = blockIdx.x * 8 + c;
    __shared__ double red[2][32][8];
    double sse = 0.0, sae = 0.0;
    if (k < K) {
        const double b0 = icpt ? icpt[k] : 0.0;
        for (long long i = (long long)blockIdx.y * 32 + r; i < m; i += (long long)SCORE_RB * 32) {
            const double* row = Xa + (GATHER ? (long long)ridx[i] : r0 + i) * lda;
            double d = row[p] - yhat[i * ldz + k] - b0 * row[p + 1];
            // rows packed as sqrt(sw_i) [x_i, y_i, 1]: the scorer wants the unweighted residual
            if (rows_scaled) d /= row[p + 1];
            sse += d * d;
            sae += fabs(d);
        }
    }
    red[0][r][c] = sse;
    red[1][r][c] = sae;
    __syncthreads();
    for (int s = 16; s > 0; s >>= 1) {
        if (r < s) {
            red[0][r][c] += red[0][r + s][c];
            red[1][r][c] += red[1][r + s][c];
        }
        __syncthreads();
    }
    if (r == 0 && k < K) {
        part[((long long)blockIdx.y * 2 + 0) * ldz + k] = red[0][0][c];
        part[((long long)blockIdx.y * 2 + 1) * ldz + k] = red[1][0][c];
    }
}
__global__ void score_final_kernel(const double* __restrict__ part, long long ldz, int K,
                                   double* __restrict__ out) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    double sse = 0.0, sae = 0.0;
    for (int b = 0; b < SCORE_RB; ++b) {
        sse += part[((long long)b * 2 + 0) * ldz + k];
        sae += part[((long long)b * 2 + 1) * ldz + k];
    }
    out[k] = sse;
    out[ldz + k] = sae;
}

// K10b (slm_cv_score_stats): residual statistics beyond the two sums, for the problem table of one scoring batch.
// They run after score_final_kernel, so the partial-sum rows of every scratch are free again.
struct StatProblem {
    double* yhat;         // [m][ldy]: predictions in, residuals out; [2 * SCORE_RB][ldy] partials from row m
    const int* ridx;      // row list, or NULL: rows r0 + i
    const double* icpt;   // [K] or NULL
    double* out;          // [5][ldy]
    long long r0, m, ldy;
    int K;
};
struct StatTable {
    StatProblem pr[kMaxGemmProblems];
};

// grid (ceil(K_max / 8), SCORE_RB, problems): the residual of score_partial_kernel replaces the prediction, and the
// block writes its partial max |r| (as bits: for non-negative doubles the bit pattern orders like the value, and a
// NaN sorts above +inf) and its partial sum of |r| / max(|y|, eps), same row split and tree as the residual sums
__global__ void __launch_bounds__(256) stat_residual_kernel(const double* __restrict__ Xa, long long lda, int p,
                                                            int rows_scaled, const __grid_constant__ StatTable t) {
    const StatProblem& q = t.pr[blockIdx.z];
    if ((int)blockIdx.x * 8 >= q.K) return;
    const int c = threadIdx.x & 7, r = threadIdx.x >> 3;
    const int k = blockIdx.x * 8 + c;
    __shared__ unsigned long long rmax[32][8];
    __shared__ double rpct[32][8];
    unsigned long long amax = 0;
    double pct = 0.0;
    if (k < q.K) {
        const double b0 = q.icpt ? q.icpt[k] : 0.0;
        for (long long i = (long long)blockIdx.y * 32 + r; i < q.m; i += (long long)SCORE_RB * 32) {
            const double* row = Xa + (q.ridx ? (long long)q.ridx[i] : q.r0 + i) * lda;
            double* yh = q.yhat + i * q.ldy + k;
            double d = row[p] - *yh - b0 * row[p + 1];
            double yv = row[p];
            if (rows_scaled) {
                d /= row[p + 1];
                yv /= row[p + 1];
            }
            *yh = d;
            const double a = fabs(d);
            amax = max(amax, (unsigned long long)__double_as_longlong(a));
            pct += a / fmax(fabs(yv), DBL_EPSILON);
        }
    }
    rmax[r][c] = amax;
    rpct[r][c] = pct;
    __syncthreads();
    for (int s = 16; s > 0; s >>= 1) {
        if (r < s) {
            rmax[r][c] = max(rmax[r][c], rmax[r + s][c]);
            rpct[r][c] += rpct[r + s][c];
        }
        __syncthreads();
    }
    if (r == 0 && k < q.K) {
        unsigned long long* part = reinterpret_cast<unsigned long long*>(q.yhat + q.m * q.ldy);
        part[((long long)blockIdx.y * 2 + 0) * q.ldy + k] = rmax[0][c];
        reinterpret_cast<double*>(part)[((long long)blockIdx.y * 2 + 1) * q.ldy + k] = rpct[0][c];
    }
}
// grid (ceil(K_max / 128), problems): out rows 2 (max |r|) and 3 (percentage sum), fixed order over the row blocks
__global__ void stat_final_kernel(int stats, const __grid_constant__ StatTable t) {
    const StatProblem& q = t.pr[blockIdx.y];
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= q.K) return;
    const double* part = q.yhat + q.m * q.ldy;
    unsigned long long amax = 0;
    double pct = 0.0;
    for (int b = 0; b < SCORE_RB; ++b) {
        amax = max(amax, reinterpret_cast<const unsigned long long*>(part)[(long long)b * 2 * q.ldy + k]);
        pct += part[((long long)b * 2 + 1) * q.ldy + k];
    }
    if (stats & SLM_STAT_MAX) q.out[2 * q.ldy + k] = __longlong_as_double((long long)amax);
    if (stats & SLM_STAT_MAPE) q.out[3 * q.ldy + k] = pct;
}

// grid (ceil(K_max / 8), problems): exact median of |r| per column by a most-significant-digit-first radix select on
// the bit patterns (8 passes of 8-bit digits), the two middle order statistics at once.  A block owns 8 adjacent
// columns (64-byte row segments); thread (c, r) reads column c of rows r, r + 32, ...; warp w finds column w's digits.
constexpr int MED_UNROLL = 4;
__global__ void __launch_bounds__(256) stat_median_kernel(const __grid_constant__ StatTable t) {
    const StatProblem& q = t.pr[blockIdx.y];
    if ((int)blockIdx.x * 8 >= q.K) return;
    const int c = threadIdx.x & 7, r = threadIdx.x >> 3, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int k = blockIdx.x * 8 + c;
    const bool col = k < q.K;
    __shared__ unsigned int hist[2][8][256];
    __shared__ unsigned long long pfx[2][8];  // digits of the two order statistics found so far
    __shared__ long long rnk[2][8];           // their ranks among the values that share that prefix
    __shared__ int has_nan[8];
    for (int j = threadIdx.x; j < 2 * 8 * 256; j += 256) (&hist[0][0][0])[j] = 0u;
    if (threadIdx.x < 16) {
        const int tt = threadIdx.x >> 3, cc = threadIdx.x & 7;
        pfx[tt][cc] = 0ull;
        rnk[tt][cc] = tt == 0 ? (q.m - 1) / 2 : q.m / 2;  // np.median: ranks (m-1)/2 and m/2
    }
    if (threadIdx.x < 8) has_nan[threadIdx.x] = 0;
    __syncthreads();
    for (int shift = 56; shift >= 0; shift -= 8) {
        const unsigned long long hmask = shift == 56 ? 0ull : ~0ull << (shift + 8);
        const unsigned long long p0 = pfx[0][c], p1 = pfx[1][c];
        // the trip count is uniform over a warp (its 4 row lanes share i0): every lane takes part in the matches
        for (long long i0 = 0; i0 < q.m; i0 += 32 * MED_UNROLL) {
            unsigned long long v[MED_UNROLL];
            bool ok[MED_UNROLL];
#pragma unroll
            for (int u = 0; u < MED_UNROLL; ++u) {
                const long long i = i0 + r + 32 * u;
                ok[u] = col && i < q.m;
                v[u] = ok[u] ? (unsigned long long)__double_as_longlong(fabs(q.yhat[i * q.ldy + k])) : 0ull;
            }
#pragma unroll
            for (int u = 0; u < MED_UNROLL; ++u) {
                const unsigned dig = (unsigned)(v[u] >> shift) & 255u;
#pragma unroll
                for (int tt = 0; tt < 2; ++tt) {
                    const bool in = ok[u] && (v[u] & hmask) == (tt ? p1 : p0);
                    // lanes adding to the same bin add once (ties and all-equal columns would serialise otherwise)
                    const unsigned key = in ? ((unsigned)c << 8 | dig) : 0xffffffffu;
                    const unsigned peers = __match_any_sync(0xffffffffu, key);
                    if (in && lane == __ffs(peers) - 1) atomicAdd(&hist[tt][c][dig], (unsigned)__popc(peers));
                }
                if (shift == 56 && ok[u] && v[u] > 0x7ff0000000000000ull) has_nan[c] = 1;
            }
        }
        __syncthreads();
        if (blockIdx.x * 8 + w < q.K) {
            for (int tt = 0; tt < 2; ++tt) {
                const unsigned int* h = hist[tt][w];
                unsigned long long s = 0;
                for (int j = 0; j < 8; ++j) s += h[lane * 8 + j];
                unsigned long long incl = s;
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned long long x = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += x;
                }
                const unsigned long long excl = incl - s;
                const long long R = rnk[tt][w];
                __syncwarp();
                if ((unsigned long long)R >= excl && (unsigned long long)R < incl) {
                    unsigned long long cum = excl;
                    int b = lane * 8;
                    while (b < lane * 8 + 7 && cum + h[b] <= (unsigned long long)R) cum += h[b++];
                    pfx[tt][w] |= (unsigned long long)b << shift;
                    rnk[tt][w] = R - (long long)cum;
                }
            }
        }
        __syncthreads();
        for (int j = threadIdx.x; j < 2 * 8 * 256; j += 256) (&hist[0][0][0])[j] = 0u;
        __syncthreads();
    }
    if (col && r == 0) {
        const double a = __longlong_as_double((long long)pfx[0][c]), b = __longlong_as_double((long long)pfx[1][c]);
        q.out[4 * q.ldy + k] = has_nan[c] ? __longlong_as_double(0x7ff8000000000000ll) : ((q.m & 1) ? a : (a + b) / 2);
    }
}

__global__ void __launch_bounds__(256) intercept_kernel(const double* __restrict__ G, long long pa, int p,
                                                        const double* __restrict__ B, long long ldz, int K,
                                                        double* __restrict__ icpt) {
    const int c = threadIdx.x & 7, r = threadIdx.x >> 3;
    const int k = blockIdx.x * 8 + c;
    __shared__ double red[32][8];
    const double* ones = G + (long long)(p + 1) * pa;
    double acc = 0.0;
    if (k < K)
        for (int j = r; j < p; j += 32) acc += ones[j] * B[(long long)j * ldz + k];
    red[r][c] = acc;
    __syncthreads();
    for (int s = 16; s > 0; s >>= 1) {
        if (r < s) red[r][c] += red[r + s][c];
        __syncthreads();
    }
    if (r == 0 && k < K) {
        const double n = ones[p + 1];
        icpt[k] = (ones[p] - red[0][c]) / n;
    }
}

// ------------------------------------------------------------------------- //
// C ABI
// ------------------------------------------------------------------------- //
extern "C" {

int slm_version(void) { return 1; }

int64_t slm_padded_cols(int64_t p) { return round_up(p + 2, 8); }

int slm_create(int device, slm_ctx** out) {
    if (!out) return 1;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return 2;  // no CUDA device: fail loudly, no fallback
    if (device < 0 || device >= ndev) return 3;
    if (cudaSetDevice(device) != cudaSuccess) return 4;
    slm_ctx* ctx = new slm_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete ctx;
        return 5;
    }
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* e = getenv("SLM_FORCE_APPLY_SHAPE")) ctx->force_apply_shape = atoi(e);
    if (const char* e = getenv("SLM_FORCE_SYRK_SHAPE")) ctx->force_syrk_shape = atoi(e);
    if (const char* e = getenv("SLM_FORCE_SPARSE_SHAPE")) ctx->force_sparse_shape = atoi(e);
    if (const char* e = getenv("SLM_COOP")) ctx->coop = atoi(e) != 0;
    if (const char* e = getenv("SLM_TRACE")) ctx->trace = atoi(e) != 0;
    if (const char* e = getenv("SLM_TMA")) ctx->tma_mask = atoi(e);
    if (const char* e = getenv("SLM_FUSED_PROX")) ctx->fused_prox = atoi(e) != 0;
    {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            ctx->encode = fn;
        else
            cudaGetLastError();
    }
    ctx->coop_max_smem = (int)prop.sharedMemPerBlockOptin;
    if (!prop.cooperativeLaunch) ctx->coop = false;
    if (cudaFuncSetAttribute(fista_coop_kernel<true, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) !=
            cudaSuccess ||
        cudaFuncSetAttribute(fista_coop_kernel<false, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) !=
            cudaSuccess) {
        cudaGetLastError();
        ctx->max_cluster = 8;
    }
    ctx->n_flags_cap = 1 << 20;
    if (cudaMalloc(&ctx->d_flags, sizeof(int) * (size_t)ctx->n_flags_cap) != cudaSuccess ||
        cudaMalloc(&ctx->d_counter, sizeof(int) * SLM_MAX_FOLDS) != cudaSuccess ||
        cudaMalloc(&ctx->d_stat, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMallocHost(&ctx->h_stat, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMalloc(&ctx->d_ratio, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMallocHost(&ctx->h_ratio, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMallocHost(&ctx->h_scount, sizeof(int) * kMaxScount) != cudaSuccess ||
        cudaMallocHost(&ctx->h_scal, sizeof(double) * 8) != cudaSuccess ||
        cudaMallocHost(&ctx->h_counter, sizeof(int) * SLM_MAX_FOLDS) != cudaSuccess) {
        delete ctx;
        return 6;
    }
    *out = ctx;
    return 0;
}

void slm_destroy(slm_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (auto& F : ctx->fam) {
        for (auto e : F.ev) cudaEventDestroy(e);
        for (auto e : F.pool) cudaEventDestroy(e);
    }
    if (ctx->d_counter) cudaFree(ctx->d_counter);
    if (ctx->d_stat) cudaFree(ctx->d_stat);
    if (ctx->h_stat) cudaFreeHost(ctx->h_stat);
    if (ctx->d_ratio) cudaFree(ctx->d_ratio);
    if (ctx->h_ratio) cudaFreeHost(ctx->h_ratio);
    if (ctx->h_scount) cudaFreeHost(ctx->h_scount);
    if (ctx->h_scal) cudaFreeHost(ctx->h_scal);
    if (ctx->d_flags) cudaFree(ctx->d_flags);
    if (ctx->h_counter) cudaFreeHost(ctx->h_counter);
    if (ctx->d_colmax) cudaFree(ctx->d_colmax);
    delete ctx;
}

int slm_set_option(slm_ctx* ctx, const char* name, int value) {
    if (!ctx || !name) return 1;
    const std::string nm(name);
    if (nm == "coop")
        ctx->coop = value != 0;
    else if (nm == "tma")
        ctx->tma_mask = value;
    else if (nm == "fused_prox")
        ctx->fused_prox = value != 0;
    else if (nm == "force_apply_shape")
        ctx->force_apply_shape = value;
    else if (nm == "force_sparse_shape")
        ctx->force_sparse_shape = value;
    else if (nm == "force_syrk_shape")
        ctx->force_syrk_shape = value;
    else
        return fail(ctx, 1, "slm_set_option: unknown option " + nm);
    return 0;
}

const char* slm_last_error(const slm_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
int slm_sm_count(const slm_ctx* ctx) { return ctx ? ctx->sm_count : 0; }
int64_t slm_launch_count(const slm_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t slm_tma_launch_count(const slm_ctx* ctx) { return ctx ? ctx->tma_launches : 0; }

int slm_timing_enable(slm_ctx* ctx, int on) {
    if (!ctx) return 1;
    ctx->timing = on != 0;
    return 0;
}
static void timing_collect(slm_ctx* ctx) {
    for (auto& F : ctx->fam) {
        for (size_t i = 0; i + 1 < F.ev.size(); i += 2) {
            float ms = 0.f;
            cudaEventSynchronize(F.ev[i + 1]);
            if (cudaEventElapsedTime(&ms, F.ev[i], F.ev[i + 1]) == cudaSuccess) F.ms += ms;
            F.pool.push_back(F.ev[i]);
            F.pool.push_back(F.ev[i + 1]);
        }
        F.ev.clear();
    }
}
int slm_timing_read(slm_ctx* ctx, int which, double* total_ms, int64_t* launches, double* flops) {
    if (!ctx || which < 0 || which >= FAM_COUNT) return 1;
    timing_collect(ctx);
    if (total_ms) *total_ms = ctx->fam[which].ms;
    if (launches) *launches = ctx->fam[which].n;
    if (flops) *flops = ctx->fam[which].flops;
    return 0;
}
int slm_apply_stats(slm_ctx* ctx, double* executed_flops, double* dense_flops) {
    if (!ctx) return 1;
    if (executed_flops) *executed_flops = ctx->apply_exec_flops;
    if (dense_flops) *dense_flops = ctx->apply_dense_flops;
    return 0;
}
int slm_timing_reset(slm_ctx* ctx) {
    if (!ctx) return 1;
    ctx->apply_exec_flops = ctx->apply_dense_flops = 0.0;
    timing_collect(ctx);
    for (auto& F : ctx->fam) {
        F.ms = 0.0;
        F.flops = 0.0;
        F.n = 0;
    }
    return 0;
}

int slm_pack_design(slm_ctx* ctx, const double* X, int64_t ldx, const double* y, const double* sw,
                    const int32_t* col_perm, const int64_t* row_perm, int64_t n, int64_t p, double* Xa,
                    int64_t lda, void* stream) {
    if (!ctx || !X || !y || !Xa) return fail(ctx, 1, "slm_pack_design: null argument");
    if (lda < p + 2 || (lda & 1)) return fail(ctx, 1, "slm_pack_design: lda must be even and >= p+2");
    if (n <= 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    int bx = (int)std::min<int64_t>((lda + 255) / 256, 64);
    for (int64_t r0 = 0; r0 < n; r0 += 65535) {  // gridDim.y limit
        int64_t nr = std::min<int64_t>(65535, n - r0);
        dim3 grid(bx, (unsigned)nr);
        // row r of this chunk is global row r0 + r
        pack_design_kernel<<<grid, 256, 0, s>>>(X + (row_perm ? 0 : r0 * ldx), ldx, y + (row_perm ? 0 : r0),
                                                sw ? sw + (row_perm ? 0 : r0) : nullptr, col_perm,
                                                row_perm ? (const long long*)(row_perm + r0) : nullptr, nr,
                                                (int)p, Xa + r0 * lda, lda);
        LAUNCH_OK("pack_design_kernel");
    }
    return 0;
}

static int gram_blocks_impl(slm_ctx* ctx, const double* Xa, int64_t lda, const int64_t* row_ptr, int n_blocks,
                            double* Gblk, int accumulate, void* stream);

int slm_gram_blocks(slm_ctx* ctx, const double* Xa, int64_t lda, const int64_t* row_ptr, int n_blocks,
                    double* Gblk, void* stream) {
    return gram_blocks_impl(ctx, Xa, lda, row_ptr, n_blocks, Gblk, 0, stream);
}

int slm_gram_block_add(slm_ctx* ctx, const double* Xa, int64_t lda, int64_t r0, int64_t r1, double* G,
                       void* stream) {
    if (r1 <= r0) return 0;
    const int64_t ptr[2] = {r0, r1};
    return gram_blocks_impl(ctx, Xa, lda, ptr, 1, G, 1, stream);
}

static int gram_blocks_impl(slm_ctx* ctx, const double* Xa, int64_t lda, const int64_t* row_ptr, int n_blocks,
                            double* Gblk, int accumulate, void* stream) {
    if (!ctx || !Xa || !row_ptr || !Gblk) return fail(ctx, 1, "slm_gram_blocks: null argument");
    if (lda % 8) return fail(ctx, 1, "slm_gram_blocks: lda must be a multiple of 8");
    cudaStream_t s = (cudaStream_t)stream;
    int sid = ctx->force_syrk_shape >= 0 && ctx->force_syrk_shape < kNumSyrkShapes ? ctx->force_syrk_shape : 0;
    for (int f0 = 0; f0 < n_blocks; f0 += kMaxGemmProblems) {
        int nf = std::min(n_blocks - f0, (int)kMaxGemmProblems);
        GemmBatch b;
        memset(&b, 0, sizeof(b));
        b.n_problems = nf;
        b.accumulate = accumulate;
        b.baseP = b.baseQ = Xa;
        b.rowsP = b.rowsQ = row_ptr[n_blocks];
        double flops = 0.0;
        for (int i = 0; i < nf; ++i) {
            int f = f0 + i;
            GemmProblem& pr = b.pr[i];
            int64_t r0 = row_ptr[f], r1 = row_ptr[f + 1];
            pr.P = pr.Q = Xa + r0 * lda;
            pr.C = Gblk + (int64_t)f * lda * lda;
            pr.ldp = pr.ldq = pr.ldc = lda;
            pr.M = pr.N = (int)lda;
            pr.Kd = (int)(r1 - r0);
            flops += (double)(r1 - r0) * (double)lda * (double)(lda + 1);  // SYRK count
        }
        FamTimer tm(ctx, FAM_GRAM, s, flops);
        cudaError_t e = launch_syrk_shape(ctx, sid, b, s);
        if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("gram build: ") + cudaGetErrorString(e));
        ctx->launches++;
    }
    return 0;
}

int slm_gram_rows_update(slm_ctx* ctx, const double* Xa, int64_t n, int64_t lda, int n_problems, const int64_t* row_ptr,
                         const int32_t* rows, double* G, int64_t g_stride, int accumulate, int negate, void* stream) {
    if (!ctx || !Xa || !row_ptr || !G) return fail(ctx, 1, "slm_gram_rows_update: null argument");
    if (lda % 8) return fail(ctx, 1, "slm_gram_rows_update: lda must be a multiple of 8");
    if (n_problems < 0 || g_stride < lda * lda) return fail(ctx, 1, "slm_gram_rows_update: bad problem count or stride");
    cudaStream_t s = (cudaStream_t)stream;
    int i = 0;
    while (i < n_problems) {
        GemmBatch b;
        memset(&b, 0, sizeof(b));
        b.accumulate = accumulate != 0;
        b.negate = negate != 0;
        b.baseP = b.baseQ = Xa;
        b.rowsP = b.rowsQ = n;
        double flops = 0.0;
        int np = 0;
        for (; i < n_problems && np < kMaxGemmProblems; ++i) {
            const int64_t m = row_ptr[i + 1] - row_ptr[i];
            if (m < 0 || m > (1LL << 30)) return fail(ctx, 1, "slm_gram_rows_update: bad row list length");
            if (m == 0) continue;  // an empty list leaves its Gram untouched
            if (!rows) return fail(ctx, 1, "slm_gram_rows_update: null row lists");
            GemmProblem& pr = b.pr[np++];
            pr.P = pr.Q = Xa;
            pr.kidx = rows + row_ptr[i];
            pr.C = G + (int64_t)i * g_stride;
            pr.ldp = pr.ldq = pr.ldc = lda;
            pr.M = pr.N = (int)lda;
            pr.Kd = (int)m;
            flops += (double)m * (double)lda * (double)(lda + 1);  // SYRK count
        }
        if (np == 0) continue;
        b.n_problems = np;
        FamTimer tm(ctx, FAM_GRAM, s, flops);
        cudaError_t e = launch_syrk_rows(ctx, b, s);
        if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("gram rows update: ") + cudaGetErrorString(e));
        ctx->launches++;
    }
    return 0;
}

int slm_gram_complement(slm_ctx* ctx, double* Gblk, int n_blocks, int64_t pa, double* Gtot, void* stream) {
    if (!ctx || !Gblk || !Gtot) return fail(ctx, 1, "slm_gram_complement: null argument");
    if (n_blocks > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_gram_complement: too many blocks");
    long long stride = (long long)pa * pa;
    gram_complement_kernel<<<(unsigned)((stride + 255) / 256), 256, 0, (cudaStream_t)stream>>>(Gblk, n_blocks,
                                                                                            stride, Gtot);
    LAUNCH_OK("gram_complement_kernel");
    return 0;
}

int64_t slm_tri_size(int64_t pa) { return pa * (pa + 1) / 2; }

int slm_tri_pack(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int n_grams, double* buf,
                 void* stream) {
    if (!ctx || !G || !buf) return fail(ctx, 1, "slm_tri_pack: null argument");
    if (n_grams <= 0 || pa <= 0) return 0;
    dim3 grid((unsigned)((pa + 255) / 256), (unsigned)pa, (unsigned)n_grams);
    tri_pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(G, g_stride, pa, buf, slm_tri_size(pa));
    LAUNCH_OK("tri_pack_kernel");
    return 0;
}

int slm_tri_unpack(slm_ctx* ctx, const double* buf, int64_t pa, int n_grams, double* G, int64_t g_stride,
                   void* stream) {
    if (!ctx || !G || !buf) return fail(ctx, 1, "slm_tri_unpack: null argument");
    if (n_grams <= 0 || pa <= 0) return 0;
    dim3 grid((unsigned)((pa + 255) / 256), (unsigned)pa, (unsigned)n_grams);
    tri_unpack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(buf, slm_tri_size(pa), pa, G, g_stride);
    LAUNCH_OK("tri_unpack_kernel");
    return 0;
}

int slm_tma_probe(slm_ctx* ctx, const double* A, int64_t rows, int64_t ld, int32_t col0, int32_t row0,
                  const int32_t* r4, double* out, void* stream) {
    if (!ctx || !A || !r4 || !out) return fail(ctx, 1, "slm_tma_probe: null argument");
    if (!ctx->encode) return fail(ctx, 8, "slm_tma_probe: cuTensorMapEncodeTiled is not available");
    CUtensorMap mt, mg;
    if (!make_map(ctx, &mt, A, rows, ld, 16) || !make_map(ctx, &mg, A, rows, ld, 1))
        return fail(ctx, 8, "slm_tma_probe: tensor map encoding failed");
    tma_probe_kernel<<<1, 128, 8192, (cudaStream_t)stream>>>(mt, mg, col0, row0, make_int4(r4[0], r4[1], r4[2], r4[3]),
                                                           out);
    LAUNCH_OK("tma_probe_kernel");
    return 0;
}

int slm_tri_complement(slm_ctx* ctx, const double* buf, int64_t pa, int n_blocks, double* G, int64_t g_stride,
                       void* stream) {
    if (!ctx || !G || !buf) return fail(ctx, 1, "slm_tri_complement: null argument");
    if (n_blocks < 1 || n_blocks > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_tri_complement: n_blocks out of range");
    if (pa <= 0) return 0;
    dim3 grid((unsigned)((pa + 255) / 256), (unsigned)pa);
    tri_complement_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(buf, slm_tri_size(pa), pa, n_blocks, G, g_stride);
    LAUNCH_OK("tri_complement_kernel");
    return 0;
}

int slm_gram_center(slm_ctx* ctx, double* G, int64_t pa, int64_t p, void* stream) {
    if (!ctx || !G) return fail(ctx, 1, "slm_gram_center: null argument");
    // NOTE: every thread reads the (unmodified) ones row; rows 0..p are updated
    dim3 grid((unsigned)((p + 1 + 255) / 256), (unsigned)(p + 1));
    gram_center_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(G, pa, (int)p);
    LAUNCH_OK("gram_center_kernel");
    return 0;
}

int slm_gram_gather(slm_ctx* ctx, const double* G, int64_t pa, int64_t p, const int32_t* idx, int64_t pe,
                    double* Ge, int64_t pae, void* stream) {
    if (!ctx || !G || !idx || !Ge) return fail(ctx, 1, "slm_gram_gather: null argument");
    if (pae < pe + 2) return fail(ctx, 1, "slm_gram_gather: pae too small");
    dim3 grid((unsigned)((pae + 255) / 256), (unsigned)pae);
    gram_gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(G, pa, (int)p, idx, (int)pe, Ge, pae);
    LAUNCH_OK("gram_gather_kernel");
    return 0;
}

int slm_gram_apply(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                   const int32_t* K, const double* Z, int64_t ldz, double* GZ, void* stream) {
    if (!ctx || !G || !K || !Z || !GZ) return fail(ctx, 1, "slm_gram_apply: null argument");
    if (ldz % 8 || pa % 2) return fail(ctx, 1, "slm_gram_apply: ldz must be a multiple of 8, pa even");
    return apply_batched(ctx, G, g_stride, pa, p, n_folds, K, Z, ldz, GZ, (cudaStream_t)stream);
}

// ---- unpenalised least squares: conjugate gradients on the Gram ------------------------
size_t slm_gram_cg_workspace(int64_t p) { return (size_t)(3 * 8 * p + p + 8) * sizeof(double); }

int slm_gram_cg(slm_ctx* ctx, const double* G, int64_t pa, int64_t p, const double* shift, double tol,
                int32_t max_iter, void* work, size_t work_bytes, double* X8, int32_t* iters_host,
                double* relres_host, void* stream) {
    if (!ctx || !G || !work || !X8) return fail(ctx, 1, "slm_gram_cg: null argument");
    if (pa % 2 || pa < p + 1) return fail(ctx, 1, "slm_gram_cg: pa must be even and hold the X^T y row");
    if (work_bytes < slm_gram_cg_workspace(p)) return fail(ctx, 1, "slm_gram_cg: workspace too small");
    if (!(tol > 0.0)) return fail(ctx, 1, "slm_gram_cg: tol must be positive");
    cudaStream_t s = (cudaStream_t)stream;
    double* D8 = (double*)work;
    double* GD8 = D8 + 8 * p;
    double* GX8 = GD8 + 8 * p;
    double* R = GX8 + 8 * p;
    double* sc = R + p;
    const int32_t K1 = 1;
    CUDA_OK(cudaMemsetAsync(work, 0, slm_gram_cg_workspace(p), s));
    CUDA_OK(cudaMemsetAsync(X8, 0, sizeof(double) * 8 * (size_t)p, s));
    cg_start_kernel<<<1, CG_T, 0, s>>>(G, pa, (int)p, X8, nullptr, shift, R, D8, sc);
    LAUNCH_OK("cg_start_kernel");
    auto scalars = [&]() -> int {  // sc -> host
        CUDA_OK(cudaMemcpyAsync(ctx->h_scal, sc, sizeof(double) * 3, cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
        return 0;
    };
    int it = 0, restarts = 0;
    double rel = 0.0;
    const int check = 8;
    while (true) {
        bool conv = false;
        for (; it < max_iter; ++it) {
            if (it % check == 0) {
                if (int rc = scalars()) return rc;
                const double rs = ctx->h_scal[0], cc = ctx->h_scal[1];
                if (!(rs == rs)) return fail(ctx, 7, "slm_gram_cg: non-finite residual");
                rel = cc > 0.0 ? sqrt(rs / cc) : 0.0;
                if (rel <= tol) {
                    conv = true;
                    break;
                }
            }
            int rc = apply_batched(ctx, G, pa * pa, pa, p, 1, &K1, D8, 8, GD8, s, -1.0, FAM_LIPS);
            if (rc) return rc;
            cg_step_kernel<<<1, CG_T, 0, s>>>((int)p, X8, R, D8, GD8, shift, sc);
            LAUNCH_OK("cg_step_kernel");
        }
        // the recurrence drifts from the true residual: recompute c - G x and, if it is not
        // there yet, restart the recurrence from x (residual replacement)
        int rc = apply_batched(ctx, G, pa * pa, pa, p, 1, &K1, X8, 8, GX8, s, -1.0, FAM_LIPS);
        if (rc) return rc;
        cg_start_kernel<<<1, CG_T, 0, s>>>(G, pa, (int)p, X8, GX8, shift, R, D8, sc);
        LAUNCH_OK("cg_start_kernel");
        if (int rc2 = scalars()) return rc2;
        rel = ctx->h_scal[1] > 0.0 ? sqrt(ctx->h_scal[0] / ctx->h_scal[1]) : 0.0;
        if (rel <= 4.0 * tol || it >= max_iter || (conv && ++restarts > 3)) break;
    }
    if (iters_host) *iters_host = it;
    if (relres_host) *relres_host = rel;
    return 0;
}

size_t slm_rowsparse_workspace(int64_t p, int64_t ldz, int n_folds) {
    size_t nblk = (size_t)ldz / 8;
    return (size_t)n_folds * nblk * ((size_t)p + 1) * sizeof(int) + (size_t)n_folds * (size_t)p * nblk + 64;
}

int slm_gram_apply_rowsparse(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                             const int32_t* K, const double* Z, int64_t ldz, double* GZ, int chunk_w, void* work,
                             size_t work_bytes, void* stream) {
    if (!ctx || !G || !K || !Z || !GZ || !work) return fail(ctx, 1, "slm_gram_apply_rowsparse: null argument");
    if (ldz % 8 || pa % 2) return fail(ctx, 1, "slm_gram_apply_rowsparse: ldz must be a multiple of 8, pa even");
    if (n_folds < 1 || n_folds > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_gram_apply_rowsparse: n_folds out of range");
    if (chunk_w < 8 || chunk_w % 8) return fail(ctx, 1, "slm_gram_apply_rowsparse: chunk_w must be a multiple of 8");
    if (work_bytes < slm_rowsparse_workspace(p, ldz, n_folds))
        return fail(ctx, 1, "slm_gram_apply_rowsparse: workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    const int ncc = (int)((ldz + chunk_w - 1) / chunk_w);
    SolveDev sp;
    memset(&sp, 0, sizeof(sp));
    sp.F = n_folds;
    sp.p = (int)p;
    sp.ldz = ldz;
    sp.pa = pa;
    sp.g_stride = g_stride;
    sp.G = G;
    sp.nblk = (int)(ldz / SC);
    int* sidx = (int*)work;
    int* scount = sidx + (size_t)n_folds * ncc * p;
    sp.zflag = (unsigned char*)(sidx + (size_t)n_folds * sp.nblk * (p + 1));
    for (int f = 0; f < n_folds; ++f) {
        if (K[f] < 0 || K[f] > ldz) return fail(ctx, 1, "slm_gram_apply_rowsparse: K[f] out of range");
        sp.K[f] = K[f];
    }
    const dim3 zgrid((unsigned)(((long long)p * sp.nblk + 255) / 256), (unsigned)n_folds);
    zflags_kernel<<<zgrid, 256, 0, s>>>(sp, Z);
    LAUNCH_OK("zflags_kernel");
    return apply_rowsparse(ctx, sp, K, Z, GZ, chunk_w, ncc, sidx, scount, s, -1.0);
}

size_t slm_lipschitz_workspace(int64_t p, int n_grams) {
    return (size_t)(2 * (int64_t)n_grams * p * 8 + n_grams) * sizeof(double);
}

// block power iteration; leaves lam[n_grams] (largest Rayleigh quotient) in the workspace
static int lipschitz_run(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_grams,
                         int iters, void* work, double** lam_out, cudaStream_t s) {
    double* V = (double*)work;
    double* W = V + (int64_t)n_grams * p * 8;
    double* lam = W + (int64_t)n_grams * p * 8;
    std::vector<int32_t> K(n_grams, 8);
    power_norm_kernel<<<n_grams, 8 * PN_LANES, 0, s>>>(V, W, (int)p, lam, 1);
    LAUNCH_OK("power_norm_kernel(init)");
    for (int it = 0; it < iters; ++it) {
        int rc = apply_batched(ctx, G, g_stride, pa, p, n_grams, K.data(), V, 8, W, s, -1.0, FAM_LIPS);
        if (rc) return rc;
        power_norm_kernel<<<n_grams, 8 * PN_LANES, 0, s>>>(V, W, (int)p, lam, 0);
        LAUNCH_OK("power_norm_kernel");
    }
    *lam_out = lam;
    return 0;
}

int slm_lipschitz(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_grams,
                  int iters, void* work, double* lam_host, void* stream) {
    if (!ctx || !G || !work || !lam_host) return fail(ctx, 1, "slm_lipschitz: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    double* lam = nullptr;
    int rc = lipschitz_run(ctx, G, g_stride, pa, p, n_grams, iters, work, &lam, s);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(lam_host, lam, sizeof(double) * n_grams, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    return 0;
}

int slm_lipschitz_dev(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_grams,
                      int iters, void* work, double* lam_dev, void* stream) {
    if (!ctx || !G || !work || !lam_dev) return fail(ctx, 1, "slm_lipschitz_dev: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    double* lam = nullptr;
    int rc = lipschitz_run(ctx, G, g_stride, pa, p, n_grams, iters, work, &lam, s);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(lam_dev, lam, sizeof(double) * n_grams, cudaMemcpyDeviceToDevice, s));
    return 0;
}

// ---- batched solve (slm_solve_batch) -------------------------------------------------------------
constexpr int kChunkW = 32;  // columns per support chunk of the row-sparse apply (its narrow form)

// byte offsets into the solve workspace: slm_solve_workspace sizes it, slm_solve_batch carves it up
struct SolveLayout {
    size_t Z, GZ, GB, T, Bw;         // [F][p][ldz] doubles each
    size_t theta, tmom, rst, part;   // doubles: [2][F][ldz], [2][F][ldz], [F][ldz], [F][kMaxChunks][NQ][ldz]
    size_t flag, colmap, src, newK;  // ints: [F][ldz] each, newK 64
    size_t sidx, scount;             // support lists [F][ncc][p] and their lengths [F][ncc] (ncc chunks of kChunkW)
    size_t zflag;                    // [F][p][ldz / 8] bytes
    size_t bytes;
};

static SolveLayout solve_layout(int64_t p, int64_t ldz, int F) {
    const size_t state = (size_t)F * p * ldz * sizeof(double), cols = (size_t)F * ldz;
    const size_t nblk = (size_t)ldz / 8, ncc = (size_t)((ldz + kChunkW - 1) / kChunkW);
    SolveLayout L;
    L.Z = 0;
    L.GZ = L.Z + state;
    L.GB = L.GZ + state;
    L.T = L.GB + state;
    L.Bw = L.T + state;
    L.theta = L.Bw + state;
    L.tmom = L.theta + 2 * cols * sizeof(double);
    L.rst = L.tmom + 2 * cols * sizeof(double);
    L.part = L.rst + cols * sizeof(double);
    L.flag = L.part + cols * kMaxChunks * NQ * sizeof(double);
    L.colmap = L.flag + cols * sizeof(int);
    L.src = L.colmap + cols * sizeof(int);
    L.newK = L.src + cols * sizeof(int);
    L.sidx = L.newK + 64 * sizeof(int);
    L.scount = L.sidx + (size_t)F * ncc * p * sizeof(int);
    L.zflag = L.sidx + (size_t)F * nblk * (p + 1) * sizeof(int);  // room for the lists of 8-column chunks
    L.bytes = L.zflag + round_up((int64_t)((size_t)F * p * nblk), 16) + 64 + 256;  // + 320 bytes of slack
    return L;
}

size_t slm_solve_workspace(int64_t p, int64_t ldz, int n_folds, int /*n_groups*/) {
    return solve_layout(p, ldz, n_folds).bytes;
}

// One slm_solve_batch call.  An iteration is a stretch (small, coop and cluster modes: every iteration up to the
// next check in one launch) or apply, check (when scheduled), prox, compact (after a check that retired columns)
// and the hand-over to the cluster kernels.  finish scatters the coefficients and certifies them.
struct BatchSolve {
    slm_ctx* const ctx;
    slm_batch* const bt;
    const cudaStream_t s;
    const int F = bt->n_folds;
    const int64_t p = bt->p, ldz = bt->ldz;
    const size_t state = (size_t)F * p * ldz;  // elements of one [F][p][ldz] array
    const bool grouped = bt->gptr_dev != nullptr;
    // small designs: the iterations between two convergence checks run inside one kernel (fista_small_kernel,
    // Gram in shared memory) and the checks use the dense apply; larger designs use the row-sparse apply
    const bool small = p <= kSmallPMax, sparse = !small;
    const int ncc = (int)((ldz + kChunkW - 1) / kChunkW);  // support chunks of kChunkW columns per fold
    const int check_every = std::max(1, bt->check_every);
    const int cw_wide = (int)std::min<int64_t>(ldz, 128);  // columns per chunk of the wide row-sparse apply
    int *colmap = nullptr, *src = nullptr, *newK = nullptr, *sidx = nullptr, *scount = nullptr;
    SolveDev sp = {};  // the arrays Z, GZ, GB, T, B (Bw), part of the workspace; K: current column counts
    int n_active_f[SLM_MAX_FOLDS] = {0};
    int Kmax0 = 0, Kmax = 0;
    long long Ktot = 0, n_active = 0;
    dim3 cgrid, mgrid, fgrid, zgrid;
    // coop: few columns on a large design, the whole GPU iterates on them inside one cooperative launch between
    // two checks.  clus: when few columns are left (or given), one thread-block cluster per column; columns are
    // independent, so any number of clusters (coop_kernels.cuh)
    bool coop = false, clus = false;
    CoopArgs ca = {};
    int coop_nb = 0, clus_cs_min = 0, clus_thr = 0;
    size_t coop_sm = 0;
    int p32 = 0, nsplit = 0;  // fista_small_kernel geometry
    size_t small_smem = 0;
    // fused iteration (solver_kernels.cuh, prox_fused_kernel): the iterates W_t / W_{t-1} alternate between Bw
    // and T, their Gram products between GZ and GB; Z is scratch.  One-way switch to the two-kernel state when
    // the cluster kernels take over the tail
    bool fused = false;
    double *Bc[2] = {}, *GBc[2] = {};
    int use_rst = 0;
    int it = 0;
    // stretching modes: checks get rarer while nothing converges
    int next_check = 0, prev_check = 0, interval = check_every;
    double prev_ratio = 0.0;
    int next_regular = 0;  // next check of the per-iteration kernels: every check_every iterations, twice
                           // as often once an eighth of the columns is left (the tail iterates at the
                           // latency floor of the launch set, a check costs about one iteration)
    bool do_compact = false;
    // chunk width of the row-sparse apply: narrow chunks (kChunkW) pay when the supports of the column chunks
    // differ, one wide chunk per fold when they are all (nearly) dense -- the narrow form then re-reads G once
    // per chunk.  Decided at every convergence check from the list lengths of that iteration (which always runs
    // narrow)
    const bool can_adapt = sparse && kChunkW < cw_wide && F * ncc <= kMaxScount;
    bool wide = false;

    BatchSolve(slm_ctx* c, slm_batch* b, cudaStream_t st) : ctx(c), bt(b), s(st) {}

    bool stretches() const { return small || coop || clus; }

    void set_grids(int K) {
        cgrid = dim3((unsigned)((K + SC - 1) / SC), (unsigned)sp.n_chunks, (unsigned)F);
        mgrid = dim3((unsigned)((K + SC - 1) / SC), (unsigned)((p + MOM_ROWS - 1) / MOM_ROWS), (unsigned)F);
        fgrid = dim3((unsigned)((K + 127) / 128), (unsigned)F);
    }

    // row-sparse apply: the row support flags of z from scratch
    int zflags(const SolveDev& d, const double* z) {
        if (!sparse) return 0;
        zflags_kernel<<<zgrid, 256, 0, s>>>(d, z);
        LAUNCH_OK("zflags_kernel");
        return 0;
    }

    // duality gaps and convergence flags of every column (final_mode: the certificate only)
    void gap_kernels(const SolveDev& d, int par, int final_mode) {
        (grouped ? gap_partial_kernel<true> : gap_partial_kernel<false>)<<<cgrid, ST, 0, s>>>(d, par, final_mode);
        gap_final_kernel<<<fgrid, 128, 0, s>>>(d, it, final_mode);
    }

    // the cooperative kernels' three beta buffers of nprob columns, in the T / GZ scratch arrays
    void coop_buffers(int nprob) {
        ca.nprob = nprob;
        ca.buf[0] = sp.T;
        ca.buf[1] = sp.T + (size_t)nprob * p;
        ca.buf[2] = sp.GZ;
        ca.dpart = sp.part;
    }

    int coop_smem_attr(bool cluster) {
        CUDA_OK(cudaFuncSetAttribute(cluster ? fista_coop_kernel<true, true> : fista_coop_kernel<true, false>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coop_sm));
        CUDA_OK(cudaFuncSetAttribute(cluster ? fista_coop_kernel<false, true> : fista_coop_kernel<false, false>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coop_sm));
        return 0;
    }

    // workspace pointers, the kernels' view of the solve, the column counts
    int init() {
        const size_t cols = (size_t)F * ldz;
        const SolveLayout L = solve_layout(p, ldz, F);
        char* w = (char*)bt->work_dev;
        colmap = (int*)(w + L.colmap);
        src = (int*)(w + L.src);
        newK = (int*)(w + L.newK);
        sidx = (int*)(w + L.sidx);
        scount = (int*)(w + L.scount);
        const int Gn = grouped ? bt->n_groups : (int)p;
        sp.F = F;
        sp.p = (int)p;
        sp.Gn = Gn;
        sp.ldz = ldz;
        sp.pa = bt->pa;
        sp.g_stride = bt->g_stride;
        sp.G = bt->G_dev;
        sp.gptr = bt->gptr_dev;
        sp.lam1 = bt->lam1_dev;
        sp.W1 = bt->W1_dev;
        sp.W2 = bt->W2_dev;
        sp.D2 = bt->D2_dev;
        sp.B = Bc[0] = (double*)(w + L.Bw);
        sp.Bout = bt->B_dev;
        sp.colmap = colmap;
        sp.skip = bt->skip_dev;
        sp.Z = (double*)(w + L.Z);
        sp.GZ = GBc[0] = (double*)(w + L.GZ);
        sp.GB = GBc[1] = (double*)(w + L.GB);
        sp.T = Bc[1] = (double*)(w + L.T);
        sp.theta[0] = (double*)(w + L.theta);
        sp.theta[1] = sp.theta[0] + cols;
        sp.tmom[0] = (double*)(w + L.tmom);
        sp.tmom[1] = sp.tmom[0] + cols;
        sp.part = (double*)(w + L.part);
        sp.rst = (double*)(w + L.rst);
        sp.flag = (int*)(w + L.flag);
        const int gpb = grouped ? GPB : SG;  // groups per block iteration
        sp.gpt = std::max(1, (Gn + gpb * kMaxChunks - 1) / (gpb * kMaxChunks));
        sp.n_chunks = (Gn + gpb * sp.gpt - 1) / (gpb * sp.gpt);
        sp.gap = bt->gap_dev;
        sp.primal = bt->primal_dev;
        sp.n_iter = bt->n_iter_dev;
        sp.status = bt->status_dev;
        sp.counter = ctx->d_counter;
        sp.ratio = ctx->d_ratio;
        sp.zflag = sparse ? (unsigned char*)(w + L.zflag) : nullptr;
        sp.nblk = (int)(ldz / SC);
        sp.tol = bt->tol;
        sp.floor_rel = bt->floor_rel;
        sp.lips_dev = bt->lipschitz_dev;
        for (int f = 0; f < F; ++f) {
            if (bt->K[f] < 0 || bt->K[f] > ldz) return fail(ctx, 1, "slm_solve_batch: K[f] out of range");
            if (bt->K[f] > 0 && ((!bt->lipschitz_dev && !(bt->lipschitz[f] > 0.0)) || !(bt->n_obs[f] > 0.0)))
                return fail(ctx, 1, "slm_solve_batch: lipschitz and n_obs must be positive");
            sp.K[f] = bt->K[f];
            sp.n_obs[f] = bt->n_obs[f] > 0.0 ? bt->n_obs[f] : 1.0;
            sp.step[f] = bt->lipschitz[f] > 0.0 ? 1.0 / bt->lipschitz[f] : 0.0;
            Kmax0 = std::max(Kmax0, bt->K[f]);
            Ktot += bt->K[f];
        }
        bt->iters_run = 0;
        bt->n_unconverged = 0;
        Kmax = Kmax0;
        n_active = Ktot;
        set_grids(Kmax);
        zgrid = dim3((unsigned)(((long long)p * sp.nblk + 255) / 256), (unsigned)F);
        return 0;
    }

    // mode choice (small, coop, cluster eligibility) and the kernel attributes the chosen mode needs
    int plan() {
        if (small) {
            p32 = (int)round_up(p, 32);
            nsplit = std::max(1, std::min(8, 256 / p32));
            small_smem = fista_small_smem((int)p, p32, nsplit);
            CUDA_OK(cudaFuncSetAttribute(fista_small_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)small_smem));
            CUDA_OK(cudaFuncSetAttribute(fista_small_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)small_smem));
            return 0;
        }
        if (!ctx->coop) return 0;
        const int maxg = grouped ? bt->max_group : 1;  // 0: the caller did not say
        coop_sm = coop_smem((int)p);
        if (maxg <= 0 || coop_sm > (size_t)ctx->coop_max_smem) return 0;
        ca.seg = coop_seg((int)p);
        if (Ktot <= kCoopMaxProb) {
            const int nprob = (int)Ktot;
            coop_nb = (int)std::min<int64_t>(ctx->sm_count / nprob, std::max<int64_t>(1, p / 16));
            if (coop_nb >= 1 && (p + coop_nb - 1) / coop_nb + maxg <= CO_ROWS) {
                coop = true;
                coop_buffers(nprob);
                int q = 0;
                for (int f = 0; f < F; ++f)
                    for (int k = 0; k < bt->K[f]; ++k, ++q) {
                        ca.pf[q] = f;
                        ca.pk[q] = k;
                    }
                return coop_smem_attr(false);
            }
        }
        if (p > 16 * CO_ROWS) return 0;
        for (int cs = 1; cs <= ctx->max_cluster; cs *= 2)
            if ((p + cs - 1) / cs + maxg <= CO_ROWS) {
                clus_cs_min = cs;
                break;
            }
        if (clus_cs_min == 0) return 0;
        // three rounds of co-resident clusters at most, and the three beta buffers of every column must fit in
        // the T / GZ scratch arrays
        clus_thr = (int)std::min<long long>(3LL * (ctx->sm_count / clus_cs_min), (long long)F * ldz / 2);
        return coop_smem_attr(true);
    }

    // initial state of every column and of the iterate buffers, the support flags
    int start() {
        const size_t cols = (size_t)F * ldz;
        init_cols_kernel<<<(unsigned)((cols + 255) / 256), 256, 0, s>>>(sp.theta[0], sp.tmom[0], sp.flag, colmap,
                                                                        sp.status, sp.n_iter, bt->skip_dev,
                                                                        (long long)cols, (int)ldz);
        LAUNCH_OK("init_cols_kernel");
        CUDA_OK(cudaMemcpyAsync(sp.B, bt->B_dev, state * sizeof(double), cudaMemcpyDeviceToDevice, s));
        CUDA_OK(cudaMemcpyAsync(sp.Z, bt->B_dev, state * sizeof(double), cudaMemcpyDeviceToDevice, s));
        CUDA_OK(cudaMemsetAsync(sp.GB, 0, state * sizeof(double), s));
        fused = ctx->fused_prox && !small && !coop;
        if (fused) CUDA_OK(cudaMemcpyAsync(sp.T, bt->B_dev, state * sizeof(double), cudaMemcpyDeviceToDevice, s));
        if (sparse) CUDA_OK(cudaMemsetAsync(ctx->d_stat, 0, sizeof(unsigned long long), s));
        return zflags(sp, sp.Z);
    }

    // small, coop and cluster modes: every iteration up to the next check (or max_iter) in one launch
    int stretch() {
        const int par = it & 1;
        int n_inner = std::min(next_check, (int)bt->max_iter) - it;
        if (clus) {
            const int nprob = (int)n_active;
            int cs = clus_cs_min;
            while (cs * 2 <= ctx->max_cluster && nprob * cs * 2 <= ctx->sm_count) cs *= 2;
            if (ctx->trace)
                fprintf(stderr, "[slm] cluster launch it=%d n_inner=%d nprob=%d cs=%d\n", it, n_inner, nprob, cs);
            coop_list_kernel<<<1, 32, 0, s>>>(sp, src);
            LAUNCH_OK("coop_list_kernel");
            coop_buffers(nprob);
            ca.plist = src;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(nprob * cs));
            cfg.blockDim = dim3(CO_T);
            cfg.dynamicSmemBytes = coop_sm;
            cfg.stream = s;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = (unsigned)cs;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            FamTimer tm(ctx, FAM_PROX, s, 0.0);
            CUDA_OK(cudaLaunchKernelEx(&cfg, grouped ? fista_coop_kernel<true, true> : fista_coop_kernel<false, true>,
                                       sp, ca, par, n_inner));
            ctx->launches++;
        } else if (coop) {
            // the SMs share the column(s), one grid barrier per iteration
            FamTimer tm(ctx, FAM_PROX, s, 0.0);
            int parv = par;
            void* args[] = {(void*)&sp, (void*)&ca, (void*)&parv, (void*)&n_inner};
            CUDA_OK(cudaLaunchCooperativeKernel(grouped ? (const void*)fista_coop_kernel<true, false>
                                                        : (const void*)fista_coop_kernel<false, false>,
                                                dim3((unsigned)coop_nb, (unsigned)ca.nprob), dim3(CO_T), args,
                                                coop_sm, s));
            ctx->launches++;
        } else {
            FamTimer tm(ctx, FAM_PROX, s, 0.0);
            (grouped ? fista_small_kernel<true> : fista_small_kernel<false>)<<<dim3((unsigned)Kmax, (unsigned)F),
                                                                             p32 * nsplit, small_smem, s>>>(
                sp, par, n_inner, p32, nsplit);
            LAUNCH_OK("fista_small_kernel");
        }
        it += n_inner - 1;
        return 0;
    }

    // chunk-width decision from the support-list lengths of a narrow iteration (host copy in ctx->h_scount):
    // time of the narrow form (per-chunk supports, G re-read per chunk) against one wide chunk per fold
    // contracting over the largest support
    void decide_width() {
        double fw = 0.0, fn = 0.0, bw = 0.0, bn = 0.0;  // flops / G bytes, wide and narrow
        for (int f = 0; f < F; ++f) {
            const int Kp = (int)std::min<int64_t>(round_up(sp.K[f], 8), ldz);
            int smax = 0;
            for (int cc = 0; cc * kChunkW < Kp; ++cc) {
                const int sc = ctx->h_scount[f * ncc + cc];
                smax = std::max(smax, sc);
                fn += 2.0 * (double)p * sc * std::min(kChunkW, Kp - cc * kChunkW);
                bn += 8.0 * (double)p * sc;
            }
            fw += 2.0 * (double)p * smax * std::min(Kp, cw_wide) * ((Kp + cw_wide - 1) / cw_wide);
            bw += 8.0 * (double)p * smax * ((Kp + cw_wide - 1) / cw_wide);
        }
        const double tn = std::max(fn / (0.84 * 35e12), bn / 6.0e12);
        const double tw = std::max(fw / (0.776 * 35e12), bw / 6.0e12);
        wide = (fn == 0.0) || (tw < tn);
    }

    // the Gram apply of one iteration (G Z, or G W_t in the fused iteration): support-flag refresh, width probe,
    // then the row-sparse or the dense apply
    int apply(bool check) {
        const int par = it & 1;
        const double algo = 2.0 * (double)p * (double)p * (double)n_active;
        int rc;
        // the cooperative iterations do not maintain the row flags
        if ((coop || clus) && it > 0 && (rc = zflags(sp, sp.Z))) return rc;
        // the supports change fastest in the first iterations (a cold start is all-zero, then every weakly
        // penalised column fills up): re-decide the width there without waiting for the next convergence check
        const bool probe = can_adapt && !check && !coop && !clus && (it == 1 || it == 3 || it == 6);
        const int cw = (wide && !check && !probe) ? cw_wide : kChunkW;
        const double* in = fused ? Bc[par] : sp.Z;  // fused: the Gram acts on the iterate itself
        double* out = fused ? GBc[par] : sp.GZ;
        rc = sparse ? apply_rowsparse(ctx, sp, sp.K, in, out, cw, (int)((ldz + cw - 1) / cw), sidx, scount, s, algo)
                    : apply_batched(ctx, bt->G_dev, bt->g_stride, bt->pa, p, F, sp.K, in, ldz, out, s, algo);
        if (rc) return rc;
        if ((check || probe) && (can_adapt || (clus_thr > 0 && sparse && F * ncc <= kMaxScount)))
            CUDA_OK(cudaMemcpyAsync(ctx->h_scount, scount, sizeof(int) * (size_t)F * ncc, cudaMemcpyDeviceToHost, s));
        if (probe) {
            CUDA_OK(cudaStreamSynchronize(s));
            decide_width();
        }
        return 0;
    }

    // few columns left: one cluster per column pays when the columns are sparse (every cluster reads its own
    // support rows of the Gram: |S| p 8 bytes per column and iteration, nothing shared between columns) --
    // otherwise the GEMM path, which shares the Gram between the columns of a chunk, stays
    bool cluster_pays() const {
        if (n_active > clus_thr || !sparse || F * ncc > kMaxScount) return false;
        double bytes = 0.0, flops = 0.0;
        for (int f = 0; f < F; ++f) {
            const int Kp = (int)std::min<int64_t>(round_up(n_active_f[f], 8), ldz);
            for (int cc = 0; cc * kChunkW < Kp; ++cc) {
                const double sc = (double)std::min<long long>(ctx->h_scount[f * ncc + cc], p);
                const double ncol = (double)std::min(kChunkW, Kp - cc * kChunkW);
                bytes += ncol * (double)p * sc * 8.0;
                flops += 2.0 * ncol * (double)p * sc;
            }
        }
        const int conc = std::max(1, std::min(ctx->sm_count / clus_cs_min, 8 * (16 / clus_cs_min)));
        const double rounds = (double)((n_active + conc - 1) / conc);
        const double t_cl = std::max(rounds * 12e-6, bytes / 3.0e12);
        const double t_ge = 90e-6 + flops / 20e12;
        return t_cl < 0.5 * t_ge;
    }

    // convergence check after this iteration's apply: gaps and flags, active counts on the host, the cluster
    // switch, the next check, the chunk width
    int check() {
        const int par = it & 1;
        CUDA_OK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(int) * SLM_MAX_FOLDS, s));
        CUDA_OK(cudaMemsetAsync(ctx->d_ratio, 0, sizeof(unsigned long long), s));
        {
            FamTimer tm(ctx, FAM_GAP, s, 0.0);
            SolveDev spg = sp;
            if (fused) {  // B = W_t, GZ = G W_t itself
                spg.B = Bc[par];
                spg.GZ = GBc[par];
                spg.direct = 1;
            }
            gap_kernels(spg, par, 0);
            if (fused) settle_done_kernel<<<mgrid, ST, 0, s>>>(sp, Bc[par], Bc[par ^ 1]);
        }
        LAUNCH_OK("gap kernels");
        ctx->launches++;
        CUDA_OK(cudaMemcpyAsync(ctx->h_counter, ctx->d_counter, sizeof(int) * SLM_MAX_FOLDS, cudaMemcpyDeviceToHost,
                                s));
        CUDA_OK(cudaMemcpyAsync(ctx->h_ratio, ctx->d_ratio, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
        n_active = 0;
        bool shrink = false;
        for (int f = 0; f < F; ++f) {
            n_active_f[f] = ctx->h_counter[f];
            n_active += n_active_f[f];
            if (round_up(n_active_f[f], 8) < round_up(sp.K[f], 8)) shrink = true;
        }
        next_regular = it + ((n_active * 8 <= Ktot && Ktot >= 16) ? std::max(2, check_every / 2) : check_every);
        if (ctx->trace)
            fprintf(stderr, "[slm] it=%d active=%lld Kmax=%d%s\n", it, n_active, Kmax,
                    coop ? " coop" : (small ? " small" : (clus ? " cluster" : "")));
        if (n_active == 0) return 0;  // every column converged: the solve stops
        if (clus_thr > 0) {
            const bool pays = cluster_pays();
            if (pays && !clus) {
                clus = true;
                interval = check_every;
                prev_ratio = 0.0;
            } else if (!pays && clus) {
                clus = false;  // the supports filled up: back to the shared-Gram GEMM iterations
            }
        }
        do_compact = shrink && !small && !coop;  // idle CTAs of the fused kernels cost nothing: no compaction
        if (stretches()) {
            // checks at 0, c, 3c, 7c, ... (c = check_every), at most 2048 apart -- sooner when the worst
            // gap/tolerance ratio of the last two checks says the tolerance is nearer than that (linear-rate
            // extrapolation + 15 %)
            int step_to = interval;
            double ratio;
            memcpy(&ratio, ctx->h_ratio, sizeof(double));
            if (prev_ratio > 0.0 && ratio > 1.0 && ratio < prev_ratio && it > prev_check) {
                const double rate = log(prev_ratio / ratio) / (double)(it - prev_check);
                const double need = 1.15 * log(ratio) / rate + 1.0;
                if (need < (double)step_to) step_to = std::max(std::max(2, check_every / 2), (int)ceil(need));
            }
            prev_ratio = ratio;
            prev_check = it;
            next_check = it + step_to;
            interval = std::min(interval * 2, 2048);
        }
        if (can_adapt) decide_width();
        return 0;
    }

    // proximal step, momentum and restart of one iteration: fused or two-kernel
    int prox() {
        const int par = it & 1;
        {
            FamTimer tm(ctx, FAM_PROX, s, 0.0);
            if (fused) {
                FusedArgs fa;
                fa.Bcur = Bc[par];
                fa.Bnew = Bc[par ^ 1];
                fa.GBcur = GBc[par];
                fa.GBold = GBc[par ^ 1];
                fa.stash = sp.Z;
                fa.it = it;
                fa.use_rst = use_rst;
                use_rst = 0;
                // rows of the largest group per sub-lane (0: the caller did not say -> the widest instantiation;
                // longer groups take the kernel's two-pass path)
                const int rows_lane = bt->max_group > 0 ? (bt->max_group + SUB - 1) / SUB : 8;
                if (!grouped)
                    prox_fused_kernel<false, 1><<<cgrid, ST, 0, s>>>(sp, fa, par);
                else if (rows_lane <= 2)
                    prox_fused_kernel<true, 2><<<cgrid, ST, 0, s>>>(sp, fa, par);
                else if (rows_lane <= 3)
                    prox_fused_kernel<true, 3><<<cgrid, ST, 0, s>>>(sp, fa, par);
                else if (rows_lane <= 5)
                    prox_fused_kernel<true, 5><<<cgrid, ST, 0, s>>>(sp, fa, par);
                else
                    prox_fused_kernel<true, 8><<<cgrid, ST, 0, s>>>(sp, fa, par);
            } else {
                (grouped ? prox_main_kernel<true> : prox_main_kernel<false>)<<<cgrid, ST, 0, s>>>(sp, par);
                prox_momentum_kernel<<<mgrid, ST, 0, s>>>(sp, par);
            }
        }
        LAUNCH_OK("prox kernels");
        ctx->launches++;
        return 0;
    }

    // converged columns leave the batch (after this iteration's epilogue, so that GZ of the old layout is no
    // longer needed): scatter their coefficients to the caller's array, move the active columns of Z, B, GB to
    // the front
    int compact() {
        const int par = it & 1;
        SolveDev spc = sp;
        if (fused) {
            // live state after this iteration's prox: W_{t+1} (other buffer), W_t, G W_t; the restart dot of the
            // iteration is reduced per column before the columns are renumbered
            spc.Z = Bc[par ^ 1];
            spc.B = Bc[par];
            spc.GB = GBc[par];
            restart_reduce_kernel<<<fgrid, 128, 0, s>>>(sp, par);
            use_rst = 1;
        }
        compact_plan_kernel<<<F, 32, 0, s>>>(sp, src, newK);
        scatter_done_kernel<<<mgrid, ST, 0, s>>>(spc, 0);
        compact_move_kernel<<<dim3((unsigned)((p + 127) / 128), 3, (unsigned)F), 128, 0, s>>>(spc, src, newK);
        compact_cols_kernel<<<F, 32, 0, s>>>(sp, src, newK, colmap);
        LAUNCH_OK("compaction kernels");
        ctx->launches += 3;
        Kmax = 0;
        for (int f = 0; f < F; ++f) {
            sp.K[f] = n_active_f[f];
            Kmax = std::max(Kmax, sp.K[f]);
        }
        set_grids(Kmax);
        do_compact = false;
        return zflags(sp, fused ? Bc[par ^ 1] : sp.Z);  // the column blocks moved: support flags from scratch
    }

    // the cluster kernels take over from the next iteration: hand them the two-kernel state
    int hand_over() {
        const int par = it & 1, pn = par ^ 1;
        fused_to_classic_kernel<<<mgrid, ST, 0, s>>>(sp, Bc[pn], Bc[par], GBc[par], it + 1, pn, use_rst);
        LAUNCH_OK("fused_to_classic_kernel");
        use_rst = 0;
        fused = false;
        return zflags(sp, sp.Z);
    }

    // coefficients still in the working array go back to the caller's layout; then the final certificate from an
    // exact G*B, in the original column order
    int finish() {
        bt->iters_run = it;
        SolveDev spe = sp;
        if (fused) spe.B = Bc[it & 1];
        scatter_done_kernel<<<mgrid, ST, 0, s>>>(spe, 1);
        LAUNCH_OK("scatter_done_kernel");
        SolveDev fin = sp;
        fin.B = bt->B_dev;
        fin.colmap = nullptr;
        for (int f = 0; f < F; ++f) fin.K[f] = bt->K[f];
        set_grids(Kmax0);
        CUDA_OK(cudaMemcpyAsync(sp.Z, bt->B_dev, state * sizeof(double), cudaMemcpyDeviceToDevice, s));
        int rc = zflags(fin, sp.Z);
        if (rc) return rc;
        if (sparse) {
            if ((rc = apply_rowsparse(ctx, fin, bt->K, sp.Z, sp.GZ, kChunkW, ncc, sidx, scount, s, 0.0))) return rc;
            CUDA_OK(cudaMemcpyAsync(ctx->h_stat, ctx->d_stat, sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
        } else if ((rc = apply_batched(ctx, bt->G_dev, bt->g_stride, bt->pa, p, F, bt->K, sp.Z, ldz, sp.GZ, s, 0.0)))
            return rc;
        CUDA_OK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(int) * SLM_MAX_FOLDS, s));
        {
            FamTimer tm(ctx, FAM_GAP, s, 0.0);
            gap_kernels(fin, 0, 1);
        }
        LAUNCH_OK("gap kernels(final)");
        ctx->launches++;
        CUDA_OK(cudaMemcpyAsync(ctx->h_counter, ctx->d_counter, sizeof(int) * SLM_MAX_FOLDS, cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaStreamSynchronize(s));
        bt->n_unconverged = 0;
        for (int f = 0; f < F; ++f) bt->n_unconverged += ctx->h_counter[f];
        if (sparse) ctx->apply_exec_flops += 2.0 * (double)p * (double)(*ctx->h_stat);
        return 0;
    }
};

int slm_solve_batch(slm_ctx* ctx, slm_batch* bt, void* stream) {
    if (!ctx || !bt) return fail(ctx, 1, "slm_solve_batch: null argument");
    if (bt->n_folds < 1 || bt->n_folds > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_solve_batch: n_folds out of range");
    if (bt->ldz % 8) return fail(ctx, 1, "slm_solve_batch: ldz must be a multiple of 8");
    if (!bt->G_dev || !bt->B_dev || !bt->work_dev) return fail(ctx, 1, "slm_solve_batch: null device pointer");
    if (bt->work_bytes < slm_solve_workspace(bt->p, bt->ldz, bt->n_folds, bt->n_groups))
        return fail(ctx, 1, "slm_solve_batch: workspace too small");
    BatchSolve b(ctx, bt, (cudaStream_t)stream);
    int rc = b.init();
    if (rc || b.Kmax0 == 0) return rc;
    if ((rc = b.plan()) || (rc = b.start())) return rc;
    for (b.it = 0; b.it < bt->max_iter; ++b.it) {
        const bool check = b.it == (b.stretches() ? b.next_check : b.next_regular);
        if (b.stretches() && !check) {
            if ((rc = b.stretch())) return rc;
            continue;
        }
        if ((rc = b.apply(check)) || (check && (rc = b.check()))) return rc;
        if (b.n_active == 0) break;
        if ((rc = b.prox()) || (b.do_compact && (rc = b.compact())) || (b.fused && b.clus && (rc = b.hand_over())))
            return rc;
    }
    return b.finish();
}

// ---- second-order phase: one lock-step Newton step of k columns (newton_kernels.cuh) ------------
static inline int64_t nw_ldh(int64_t p) { return round_up(p, 8); }
static inline int nw_panels(int64_t p) { return (int)((p + NW_NB - 1) / NW_NB); }

size_t slm_newton_workspace(int64_t p, int32_t n_groups, int32_t k, int n_folds) {
    const size_t ldh = (size_t)nw_ldh(p), kk = (size_t)k;
    const size_t ldz = (size_t)round_up(k, 8);
    size_t d = kk * ldh * ldh;                          // H
    d += kk * (size_t)nw_panels(p) * NW_NB * NW_NB;     // inverses of the diagonal blocks
    d += 6 * kk * ldh;                                  // U, KK, DP, GS, GRAD, DIR
    d += (size_t)round_up((int64_t)(kk * (size_t)n_groups), 2);  // NRM (even: what follows stays 16-byte aligned)
    d += 2 * (size_t)n_folds * (size_t)p * ldz;         // Z, GZ of the Gram apply
    return d * sizeof(double) + (4 * kk + kk * ldh + 64) * sizeof(int) + 256;  // fold, slot, info, MS, ACT
}

// slm_newton_step is the W1 = NULL case of slm_newton_step_l1 (the kernels branch on W1 only)
static int newton_step_impl(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                            int32_t k, const int32_t* fold_host, const double* nobs_dev, double* X, const double* W2,
                            const double* D2, const double* W1, const int32_t* gptr, const int32_t* gid,
                            int32_t n_groups, void* work, size_t work_bytes, double* out, void* stream) {
    if (!ctx || !G || !fold_host || !nobs_dev || !X || !W2 || !gptr || !gid || !work || !out)
        return fail(ctx, 1, "slm_newton_step: null argument");
    if (k <= 0) return 0;
    if (n_folds < 1 || n_folds > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_newton_step: n_folds out of range");
    if (work_bytes < slm_newton_workspace(p, n_groups, k, n_folds))
        return fail(ctx, 1, "slm_newton_step: workspace too small");
    if (n_groups > 6000) return fail(ctx, 1, "slm_newton_step: too many groups for the line-search kernel");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t ldv = nw_ldh(p), ldz = round_up(k, 8);
    double* H = (double*)work;
    double* INV = H + (size_t)k * ldv * ldv;
    double* U = INV + (size_t)k * nw_panels(p) * NW_NB * NW_NB;
    double* KK = U + (size_t)k * ldv;
    double* DP = KK + (size_t)k * ldv;
    double* GS = DP + (size_t)k * ldv;
    double* GRAD = GS + (size_t)k * ldv;
    double* DIR = GRAD + (size_t)k * ldv;
    double* NRM = DIR + (size_t)k * ldv;
    double* Z = NRM + (size_t)round_up((int64_t)k * n_groups, 2);
    double* GZ = Z + (size_t)n_folds * p * ldz;
    int* fold_dev = (int*)(GZ + (size_t)n_folds * p * ldz);
    int* slot_dev = fold_dev + k;
    int* info = slot_dev + k;
    int* MS = info + k;      // active coordinates per column
    int* ACT = MS + k;       // [k][ldv] their indices, ascending

    // columns of a fold take consecutive slots of that fold's block in the apply layout
    std::vector<int32_t> fs(2 * (size_t)k), Kf(n_folds, 0);
    for (int c = 0; c < k; ++c) {
        const int f = fold_host[c];
        if (f < 0 || f >= n_folds) return fail(ctx, 1, "slm_newton_step: fold index out of range");
        fs[c] = f;
        fs[k + c] = Kf[f]++;
    }
    CUDA_OK(cudaMemcpyAsync(fold_dev, fs.data(), sizeof(int32_t) * 2 * (size_t)k, cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemsetAsync(info, 0, sizeof(int) * (size_t)k, s));
    CUDA_OK(cudaMemsetAsync(Z, 0, sizeof(double) * (size_t)n_folds * p * ldz, s));

    if (!ctx->newton_smem_set) {  // per device (a function attribute is set on the current device only)
        CUDA_OK(cudaFuncSetAttribute(chol_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NW_TILE_SMEM));
        CUDA_OK(cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NW_TILE_SMEM));
        CUDA_OK(cudaFuncSetAttribute(newton_linesearch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
        CUDA_OK(cudaFuncSetAttribute(chol_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
        ctx->newton_smem_set = true;
    }
    const dim3 vgrid((unsigned)((p + NW_T - 1) / NW_T), (unsigned)k);
    newton_prepare_kernel<<<k, NW_T, 0, s>>>((int)p, n_groups, gptr, X, ldv, W2, D2, W1, NRM, U, KK, DP, ACT, MS);
    std::vector<int> ms((size_t)k);
    CUDA_OK(cudaMemcpyAsync(ms.data(), MS, sizeof(int) * (size_t)k, cudaMemcpyDeviceToHost, s));
    newton_pack_kernel<<<vgrid, NW_T, 0, s>>>((int)p, fold_dev, slot_dev, X, ldv, Z, ldz);
    LAUNCH_OK("newton prepare/pack kernels");
    if (int rc = apply_batched(ctx, G, g_stride, pa, p, n_folds, Kf.data(), Z, ldz, GZ, s, -1.0, FAM_LIPS)) return rc;
    newton_grad_kernel<<<vgrid, NW_T, 0, s>>>((int)p, G, g_stride, pa, fold_dev, slot_dev, nobs_dev, X, GZ, ldz, ldv, KK,
                                              DP, W1, GS, GRAD);
    // the host learns the matrix sizes (the gradient's Gram apply runs meanwhile): the factorisation works on
    // the active coordinates of every column, sum_c m_c^3/3 flops instead of k p^3/3
    CUDA_OK(cudaStreamSynchronize(s));
    int m_max = 0;
    for (int c = 0; c < k; ++c) m_max = std::max(m_max, ms[c]);
    const int64_t ldh = std::max<int64_t>(8, nw_ldh(m_max));
    const int npan = std::max(1, nw_panels(m_max));
    if (m_max > 0) {
        const dim3 hgrid((unsigned)((ldh + NW_T - 1) / NW_T), (unsigned)ldh, (unsigned)k);
        newton_hessian_kernel<<<hgrid, NW_T, 0, s>>>((int)p, G, g_stride, pa, fold_dev, nobs_dev, gid, U, KK, DP, ldv, ACT, MS,
                                                     H, ldh);
    }
    LAUNCH_OK("newton grad/hessian kernels");
    ctx->launches += 3;

    // blocked Cholesky, all k matrices in lock step (a matrix that ended before the panel sits out)
    for (int pn = 0; pn < npan; ++pn) {
        const int j0 = pn * NW_NB;
        chol_diag_kernel<<<k, NW_T, NW_TILE_SMEM, s>>>(H, ldh, j0, MS, INV, npan, pn, info);
        LAUNCH_OK("chol_diag_kernel");
        const int64_t rows_max = (int64_t)m_max - j0 - NW_NB;
        if (rows_max <= 0) break;
        const dim3 pgrid((unsigned)((rows_max + NW_NB - 1) / NW_NB), (unsigned)k);
        chol_panel_kernel<<<pgrid, NW_T, NW_TILE_SMEM, s>>>(H, ldh, j0, MS, INV, npan, pn);
        LAUNCH_OK("chol_panel_kernel");
        // trailing update H22 -= U12' U12 on the tensor-core GEMM: the 64 panel rows are the K-major
        // operand as they lie in H (SYM: P == Q; negated product; upper tiles only)
        GemmBatch b;
        int np_ = 0;
        auto flush = [&]() -> int {
            if (np_ == 0) return 0;
            b.n_problems = np_;
            b.baseP = b.baseQ = H;
            b.rowsP = b.rowsQ = (int64_t)k * ldh;
            FamTimer tm(ctx, FAM_LIPS, s, 0.0);
            // TMA-fed like the Gram build (the producer warp runs ahead into the next tile's panel rows while
            // the consumers are in the epilogue of the current one); cp.async kernel when TMA is switched off
            cudaError_t e = tma_prepare(ctx, b, 1) ? launch_gemm_tma_t<2, 4, 8, 4, true, 1, false, 32, 3>(ctx, b, s)
                                                   : launch_gemm_t<2, 4, 8, 4, false, true, 1>(ctx, b, s);
            if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("newton trailing update: ") + cudaGetErrorString(e));
            ctx->launches++;
            np_ = 0;
            return 0;
        };
        for (int c = 0; c < k; ++c) {
            const int64_t off = j0 + NW_NB, rows = (int64_t)ms[c] - off;
            if (rows <= 0) continue;
            if (np_ == 0) {
                memset(&b, 0, sizeof(b));
                b.accumulate = 1;
                b.negate = 1;
                b.upper_only = 1;
            }
            GemmProblem& pr = b.pr[np_++];
            pr.P = pr.Q = H + (int64_t)c * ldh * ldh + (int64_t)j0 * ldh + off;
            pr.C = H + (int64_t)c * ldh * ldh + off * ldh + off;
            pr.ldp = pr.ldq = pr.ldc = ldh;
            pr.qlim = (int)(ldh - off);
            pr.M = pr.N = (int)round_up(rows, 2);  // an odd tail touches the (identity) padding row / column with zeros
            pr.Kd = NW_NB;
            if (np_ == kMaxGemmProblems)
                if (int rc = flush()) return rc;
        }
        if (int rc = flush()) return rc;
    }
    const size_t solve_smem = sizeof(double) * ((size_t)ldh + NW_NB + (NW_TS / 32) * NW_NB);
    if (solve_smem > 98304 || 2 * sizeof(double) * (size_t)n_groups > 98304)
        return fail(ctx, 1, "slm_newton_step: design too large for the solve / line-search kernels");
    chol_solve_kernel<<<k, NW_TS, solve_smem, s>>>(H, ldh, (int)p, ACT, MS, INV, npan, GRAD, DIR, ldv);
    newton_linesearch_kernel<<<k, NW_T, 2 * sizeof(double) * (size_t)n_groups, s>>>(
        (int)p, n_groups, gptr, X, DIR, GS, GRAD, U, KK, DP, ldv, W2, NRM, W1, info, out);
    LAUNCH_OK("newton solve / line-search kernels");
    ctx->launches += 1;
    return 0;
}

int slm_newton_step(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                    int32_t k, const int32_t* fold_host, const double* nobs_dev, double* X, const double* W2,
                    const double* D2, const int32_t* gptr, const int32_t* gid, int32_t n_groups, void* work,
                    size_t work_bytes, double* out, void* stream) {
    return newton_step_impl(ctx, G, g_stride, pa, p, n_folds, k, fold_host, nobs_dev, X, W2, D2, nullptr, gptr, gid,
                            n_groups, work, work_bytes, out, stream);
}

int slm_newton_step_l1(slm_ctx* ctx, const double* G, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                       int32_t k, const int32_t* fold_host, const double* nobs_dev, double* X, const double* W2,
                       const double* D2, const double* W1, const int32_t* gptr, const int32_t* gid, int32_t n_groups,
                       void* work, size_t work_bytes, double* out, void* stream) {
    return newton_step_impl(ctx, G, g_stride, pa, p, n_folds, k, fold_host, nobs_dev, X, W2, D2, W1, gptr, gid,
                            n_groups, work, work_bytes, out, stream);
}

int slm_adaptive_update(slm_ctx* ctx, const double* B, int64_t p, int64_t ldz, int32_t K, int32_t n_groups,
                        const int32_t* gptr, const double* gw, const double* a1, const double* a2,
                        const double* alpha, double eps, double* W1, double* W2, double* dnorm,
                        void* stream) {
    if (!ctx || !B || !alpha) return fail(ctx, 1, "slm_adaptive_update: null argument");
    if (K <= 0) return 0;
    const int Gn = gptr ? n_groups : (int)p;
    adaptive_kernel<<<(unsigned)((K + CT - 1) / CT), PT, 0, (cudaStream_t)stream>>>(
        B, (int)p, ldz, K, Gn, gptr, gw, a1, a2, alpha, eps, W1, W2, dnorm);
    LAUNCH_OK("adaptive_kernel");
    return 0;
}

int slm_fold_back(slm_ctx* ctx, const double* Be, const int32_t* inv_ptr, const int32_t* inv_idx, int64_t p,
                  int64_t ldz, int32_t K, double* coef, void* stream) {
    if (!ctx || !Be || !inv_ptr || !inv_idx || !coef) return fail(ctx, 1, "slm_fold_back: null argument");
    if (K <= 0 || p <= 0) return 0;
    dim3 grid((unsigned)((K + 127) / 128), (unsigned)p);
    fold_back_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(Be, inv_ptr, inv_idx, (int)p, ldz, K, coef);
    LAUNCH_OK("fold_back_kernel");
    return 0;
}

int slm_support_counts(slm_ctx* ctx, const double* coef, int F, int64_t p, int64_t ldz, int K, double rel_tol,
                       int32_t* counts, uint8_t* uni, void* stream) {
    if (!ctx || !coef || !counts || !uni) return fail(ctx, 1, "slm_support_counts: null argument");
    if (F < 0 || F > SLM_MAX_FOLDS || K < 0 || (int64_t)K > ldz || p < 0)
        return fail(ctx, 1, "slm_support_counts: bad shape (need 0 <= F <= SLM_MAX_FOLDS, 0 <= K <= ldz)");
    if (!(rel_tol >= 0.0 && rel_tol <= DBL_MAX)) return fail(ctx, 1, "slm_support_counts: rel_tol must be finite and >= 0");
    if (F == 0 || K == 0 || p == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t need = (size_t)F * (size_t)ldz;
    if (need > ctx->colmax_cap) {
        // growing synchronises the device (cudaFree): it happens once per larger shape
        if (ctx->d_colmax) CUDA_OK(cudaFree(ctx->d_colmax));
        ctx->d_colmax = nullptr;
        ctx->colmax_cap = 0;
        CUDA_OK(cudaMalloc(&ctx->d_colmax, need * sizeof(unsigned long long)));
        ctx->colmax_cap = need;
    }
    CUDA_OK(cudaMemsetAsync(ctx->d_colmax, 0, need * sizeof(unsigned long long), s));
    const int rows_per_block = SEL_ROWS * SEL_RPT;
    dim3 g1((unsigned)((K + 31) / 32), (unsigned)F, (unsigned)((p + rows_per_block - 1) / rows_per_block));
    support_colmax_kernel<<<g1, dim3(32, SEL_ROWS), 0, s>>>(coef, p, ldz, K, ctx->d_colmax);
    LAUNCH_OK("support_colmax_kernel");
    support_count_kernel<<<(unsigned)((p + SEL_ROWS - 1) / SEL_ROWS), dim3(32, SEL_ROWS), 0, s>>>(
        coef, F, p, ldz, K, rel_tol, ctx->d_colmax, counts, uni);
    LAUNCH_OK("support_count_kernel");
    return 0;
}

int slm_cv_score(slm_ctx* ctx, const double* Xa, int64_t lda, int64_t p, int64_t r0, int64_t r1,
                 const double* B, int64_t ldz, int32_t K, const double* icpt, int32_t rows_scaled, double* yhat,
                 double* out, void* stream) {
    if (!ctx || !Xa || !B || !yhat || !out) return fail(ctx, 1, "slm_cv_score: null argument");
    if (ldz % 8) return fail(ctx, 1, "slm_cv_score: ldz must be a multiple of 8");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t m = r1 - r0;
    if (m <= 0 || K <= 0) return 0;
    GemmBatch b;
    memset(&b, 0, sizeof(b));
    b.n_problems = 1;
    GemmProblem& pr = b.pr[0];
    pr.P = Xa + r0 * lda;
    pr.Q = B;
    pr.C = yhat;
    pr.ldp = lda;
    pr.ldq = ldz;
    pr.ldc = ldz;
    pr.M = (int)m;
    pr.N = (int)std::min<int64_t>(round_up(K, 8), ldz);
    pr.Kd = (int)p;
    ProblemDims pd = {pr.M, pr.N};
    int sid = pick_shape(kScoreShapes, kNumScoreShapes, &pd, 1, ctx->sm_count);
    {
        FamTimer tm(ctx, FAM_SCORE, s, 2.0 * (double)m * (double)p * (double)K);
        cudaError_t e = launch_score_shape(ctx, sid, b, s);
        if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("score gemm: ") + cudaGetErrorString(e));
        ctx->launches++;
    }
    double* part = yhat + m * ldz;
    dim3 grid((unsigned)((K + 7) / 8), SCORE_RB);
    score_partial_kernel<<<grid, 256, 0, s>>>(Xa, lda, (int)p, r0, m, yhat, ldz, K, icpt, rows_scaled, part);
    LAUNCH_OK("score_partial_kernel");
    score_final_kernel<<<(unsigned)((K + 127) / 128), 128, 0, s>>>(part, ldz, K, out);
    LAUNCH_OK("score_final_kernel");
    return 0;
}

// several scoring problems in one GEMM launch (the row-sharded scoring of a sharded grid holds a dozen small
// ones: a slice of every fold's rows x the columns every rank solved on that fold).  rows == NULL: problem i is the
// row range [r0[i], r1[i]); else the device row list rows[i] of n_rows[i] rows (gathered A rows in the GEMM and in
// the residual sums).  slm_cv_score_many and slm_cv_score_rows are the stats == 0 cases of slm_cv_score_stats: the
// statistics kernels run only when stats asks for them.
static int cv_score_impl(slm_ctx* ctx, const char* fn, const double* Xa, int64_t lda, int64_t p, int32_t n,
                         const int64_t* r0, const int64_t* r1, const int32_t* const* rows, const int64_t* n_rows,
                         const double* const* B, const int64_t* ldb, const int32_t* K, const double* const* icpt,
                         int32_t rows_scaled, int32_t stats, double* const* yhat, const int64_t* ldy,
                         double* const* out, void* stream) {
    if (!ctx || !Xa || (rows ? !n_rows : (!r0 || !r1)) || !B || !ldb || !K || !yhat || !ldy || !out)
        return fail(ctx, 1, std::string(fn) + ": null argument");
    if (stats & ~(3 | SLM_STAT_MAX | SLM_STAT_MAPE | SLM_STAT_MEDIAN))
        return fail(ctx, 1, std::string(fn) + ": unknown statistic in the stats mask");
    stats &= SLM_STAT_MAX | SLM_STAT_MAPE | SLM_STAT_MEDIAN;  // the two sums are always computed
    cudaStream_t s = (cudaStream_t)stream;
    auto rows_of = [&](int i) -> int64_t { return rows ? n_rows[i] : r1[i] - r0[i]; };
    for (int i0 = 0; i0 < n; i0 += kMaxGemmProblems) {
        const int nb = std::min<int>(n - i0, kMaxGemmProblems);
        GemmBatch b;
        memset(&b, 0, sizeof(b));
        ProblemDims pd[kMaxGemmProblems];
        int np = 0;
        double flops = 0.0;
        for (int i = i0; i < i0 + nb; ++i) {
            const int64_t m = rows_of(i);
            if (m <= 0 || K[i] <= 0) continue;
            if (rows && m > (1LL << 30)) return fail(ctx, 1, std::string(fn) + ": row list too long");
            if ((rows && !rows[i]) || !B[i] || !yhat[i] || !out[i] || (ldb[i] & 1) || (ldy[i] % 8) ||
                ((uintptr_t)B[i] & 15))
                return fail(ctx, 1, std::string(fn) + ": bad problem (null pointer, odd leading dimension or unaligned B)");
            GemmProblem& pr = b.pr[np];
            pr.P = rows ? Xa : Xa + r0[i] * lda;
            if (rows) pr.kidx = rows[i];
            pr.Q = B[i];
            pr.C = yhat[i];
            pr.ldp = lda;
            pr.ldq = ldb[i];
            pr.ldc = ldy[i];
            pr.M = (int)m;
            pr.N = (int)std::min<int64_t>(round_up(K[i], 8), ldy[i]);
            pr.qlim = pr.N;
            pr.Kd = (int)p;
            pd[np] = {pr.M, pr.N};
            flops += 2.0 * (double)m * (double)p * (double)K[i];
            ++np;
        }
        if (np == 0) continue;
        b.n_problems = np;
        const int sid = pick_shape(kScoreShapes, kNumScoreShapes, pd, np, ctx->sm_count);
        {
            FamTimer tm(ctx, FAM_SCORE, s, flops);
            cudaError_t e = rows ? launch_score_rows_shape(ctx, sid, b, s) : launch_score_shape(ctx, sid, b, s);
            if (e != cudaSuccess) return fail(ctx, 100 + (int)e, std::string("score gemm: ") + cudaGetErrorString(e));
            ctx->launches++;
        }
        StatTable st;
        int nst = 0, kmax = 0;
        for (int i = i0; i < i0 + nb; ++i) {
            const int64_t m = rows_of(i);
            if (m <= 0 || K[i] <= 0) continue;
            double* part = yhat[i] + m * ldy[i];
            dim3 grid((unsigned)((K[i] + 7) / 8), SCORE_RB);
            if (rows)
                score_partial_kernel<true><<<grid, 256, 0, s>>>(Xa, lda, (int)p, 0, m, yhat[i], ldy[i], K[i],
                                                                icpt ? icpt[i] : nullptr, rows_scaled, part, rows[i]);
            else
                score_partial_kernel<<<grid, 256, 0, s>>>(Xa, lda, (int)p, r0[i], m, yhat[i], ldy[i], K[i],
                                                          icpt ? icpt[i] : nullptr, rows_scaled, part);
            score_final_kernel<<<(unsigned)((K[i] + 127) / 128), 128, 0, s>>>(part, ldy[i], K[i], out[i]);
            st.pr[nst++] = {yhat[i], rows ? rows[i] : nullptr, icpt ? icpt[i] : nullptr, out[i], rows ? 0 : r0[i], m,
                            ldy[i], K[i]};
            kmax = std::max<int>(kmax, K[i]);
        }
        LAUNCH_OK("score kernels");
        if (stats == 0) continue;
        // one launch of each statistics kernel for the whole table
        stat_residual_kernel<<<dim3((unsigned)((kmax + 7) / 8), SCORE_RB, (unsigned)nst), 256, 0, s>>>(
            Xa, lda, (int)p, rows_scaled, st);
        if (stats & (SLM_STAT_MAX | SLM_STAT_MAPE))
            stat_final_kernel<<<dim3((unsigned)((kmax + 127) / 128), (unsigned)nst), 128, 0, s>>>(stats, st);
        if (stats & SLM_STAT_MEDIAN)
            stat_median_kernel<<<dim3((unsigned)((kmax + 7) / 8), (unsigned)nst), 256, 0, s>>>(st);
        LAUNCH_OK("score statistics kernels");
    }
    return 0;
}

int slm_cv_score_many(slm_ctx* ctx, const double* Xa, int64_t lda, int64_t p, int32_t n, const int64_t* r0,
                      const int64_t* r1, const double* const* B, const int64_t* ldb, const int32_t* K,
                      const double* const* icpt, int32_t rows_scaled, double* const* yhat, const int64_t* ldy,
                      double* const* out, void* stream) {
    return cv_score_impl(ctx, "slm_cv_score_many", Xa, lda, p, n, r0, r1, nullptr, nullptr, B, ldb, K, icpt,
                         rows_scaled, 0, yhat, ldy, out, stream);
}

// the same with a device row list per problem instead of a row range (arbitrary CV splits)
int slm_cv_score_rows(slm_ctx* ctx, const double* Xa, int64_t lda, int64_t p, int32_t n, const int32_t* const* rows,
                      const int64_t* n_rows, const double* const* B, const int64_t* ldb, const int32_t* K,
                      const double* const* icpt, int32_t rows_scaled, double* const* yhat, const int64_t* ldy,
                      double* const* out, void* stream) {
    if (!rows) return fail(ctx, 1, "slm_cv_score_rows: null argument");
    return cv_score_impl(ctx, "slm_cv_score_rows", Xa, lda, p, n, nullptr, nullptr, rows, n_rows, B, ldb, K, icpt,
                         rows_scaled, 0, yhat, ldy, out, stream);
}

int slm_cv_score_stats(slm_ctx* ctx, const double* Xa, int64_t lda, int64_t p, int32_t n, const int64_t* r0,
                       const int64_t* r1, const int32_t* const* rows, const int64_t* n_rows, const double* const* B,
                       const int64_t* ldb, const int32_t* K, const double* const* icpt, int32_t rows_scaled,
                       int32_t stats, double* const* yhat, const int64_t* ldy, double* const* out, void* stream) {
    return cv_score_impl(ctx, "slm_cv_score_stats", Xa, lda, p, n, r0, r1, rows, n_rows, B, ldb, K, icpt, rows_scaled,
                         stats, yhat, ldy, out, stream);
}

int slm_intercepts(slm_ctx* ctx, const double* G, int64_t pa, int64_t p, const double* B, int64_t ldz,
                   int32_t K, double* icpt, void* stream) {
    if (!ctx || !G || !B || !icpt) return fail(ctx, 1, "slm_intercepts: null argument");
    if (K <= 0) return 0;
    intercept_kernel<<<(unsigned)((K + 7) / 8), 256, 0, (cudaStream_t)stream>>>(G, pa, (int)p, B, ldz, K, icpt);
    LAUNCH_OK("intercept_kernel");
    return 0;
}

// ---- standardize=True: per-group whitening (whiten_kernels.cuh) -------------------
int slm_group_whiten_factors(slm_ctx* ctx, const double* G, int64_t pa, int64_t p, const int32_t* gptr,
                             const int64_t* wptr, int32_t n_groups, const double* shift, double* W,
                             double* scratch, int32_t* info, void* stream) {
    if (!ctx || !G || !gptr || !wptr || !W || !scratch || !info)
        return fail(ctx, 1, "slm_group_whiten_factors: null argument");
    (void)p;
    if (n_groups <= 0) return 0;
    group_chol_inv_kernel<<<(unsigned)n_groups, 256, 0, (cudaStream_t)stream>>>(
        G, pa, gptr, (const long long*)wptr, shift, W, scratch, info);
    LAUNCH_OK("group_chol_inv_kernel");
    return 0;
}

int slm_gram_whiten(slm_ctx* ctx, const double* G, int64_t pa, int64_t p, const int32_t* gptr,
                    const int64_t* wptr, int32_t n_groups, const double* W, const double* ridge,
                    double ridge_scale, double* tmp, double* Gout, void* stream) {
    if (!ctx || !G || !gptr || !wptr || !W || !tmp || !Gout) return fail(ctx, 1, "slm_gram_whiten: null argument");
    if (G == Gout || tmp == Gout || tmp == G) return fail(ctx, 1, "slm_gram_whiten: buffers must be distinct");
    if (n_groups <= 0 || p <= 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    dim3 grid((unsigned)((pa + 255) / 256), (unsigned)pa);
    whiten_left_kernel<<<grid, 256, 0, s>>>(G, pa, (int)p, gptr, (const long long*)wptr, n_groups, W, tmp);
    LAUNCH_OK("whiten_left_kernel");
    whiten_right_kernel<<<grid, 256, 0, s>>>(tmp, pa, (int)p, gptr, (const long long*)wptr, n_groups, W, ridge,
                                            ridge_scale, Gout);
    LAUNCH_OK("whiten_right_kernel");
    return 0;
}

int slm_coef_unwhiten(slm_ctx* ctx, const double* Bg, int64_t p, int64_t ldz, int32_t K, const int32_t* gptr,
                      const int64_t* wptr, int32_t n_groups, const double* W, double* B, void* stream) {
    if (!ctx || !Bg || !gptr || !wptr || !W || !B) return fail(ctx, 1, "slm_coef_unwhiten: null argument");
    if (Bg == B) return fail(ctx, 1, "slm_coef_unwhiten: in-place call not supported");
    if (K <= 0 || p <= 0) return 0;
    dim3 grid((unsigned)((K + 127) / 128), (unsigned)p);
    unwhiten_coef_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(Bg, (int)p, ldz, K, gptr, (const long long*)wptr,
                                                                n_groups, W, B);
    LAUNCH_OK("unwhiten_coef_kernel");
    return 0;
}

}  // extern "C"

// ---- collectives of the sharded search on the caller's NCCL communicator -------------------------------
// SURVEY 8b / north_star: "X row-sharded, partial Grams combined with an NCCL all-reduce", "NCCL all-gather
// of CV scores and coefficients".  The library does not link against NCCL: the entry points are looked up in
// the process (the host already loaded the NCCL its communicator belongs to -- torch's bundled one when the
// communicator comes from torch.distributed), so communicator and functions always match.
#include <dlfcn.h>
typedef int (*NcclAllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*NcclAllGatherFn)(const void*, void*, size_t, int, void*, cudaStream_t);
typedef const char* (*NcclErrFn)(int);
static void* nccl_sym(const char* name) {
    void* fn = dlsym(RTLD_DEFAULT, name);
    if (!fn) {
        static void* h = nullptr;
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (h) fn = dlsym(h, name);
    }
    return fn;
}
constexpr int kNcclFloat64 = 8, kNcclSum = 0;  // ncclDataType_t / ncclRedOp_t values of nccl.h (stable ABI)

static int nccl_fail(slm_ctx* ctx, const char* what, int rc) {
    NcclErrFn es = (NcclErrFn)nccl_sym("ncclGetErrorString");
    return fail(ctx, 200 + rc, std::string(what) + ": " + (es ? es(rc) : "NCCL error"));
}

extern "C" int slm_allreduce_sum(slm_ctx* ctx, void* nccl_comm, double* buf, int64_t count, void* stream) {
    if (!ctx || !nccl_comm || !buf) return fail(ctx, 1, "slm_allreduce_sum: null argument");
    NcclAllReduceFn ar = (NcclAllReduceFn)nccl_sym("ncclAllReduce");
    if (!ar) return fail(ctx, 9, "slm_allreduce_sum: NCCL is not loaded in this process");
    if (count <= 0) return 0;
    int rc = ar(buf, buf, (size_t)count, kNcclFloat64, kNcclSum, nccl_comm, (cudaStream_t)stream);
    if (rc) return nccl_fail(ctx, "ncclAllReduce", rc);
    ctx->launches++;
    return 0;
}

extern "C" int slm_gather_results(slm_ctx* ctx, void* nccl_comm, const double* send, double* recv,
                                  int64_t count_per_rank, void* stream) {
    if (!ctx || !nccl_comm || !send || !recv) return fail(ctx, 1, "slm_gather_results: null argument");
    NcclAllGatherFn ag = (NcclAllGatherFn)nccl_sym("ncclAllGather");
    if (!ag) return fail(ctx, 9, "slm_gather_results: NCCL is not loaded in this process");
    if (count_per_rank <= 0) return 0;
    int rc = ag(send, recv, (size_t)count_per_rank, kNcclFloat64, nccl_comm, (cudaStream_t)stream);
    if (rc) return nccl_fail(ctx, "ncclAllGather", rc);
    ctx->launches++;
    return 0;
}

extern "C" int slm_tri_complement(slm_ctx* ctx, const double* buf, int64_t pa, int n_blocks, double* G,
                                  int64_t g_stride, void* stream);

// partial fold blocks G[n_blocks][pa][pa] of this rank -> training Grams + total of ALL ranks in
// G[n_blocks + 1][pa][pa]: pack the upper triangles, one all-reduce, unpack + complement in one pass
extern "C" int slm_gram_allreduce(slm_ctx* ctx, void* nccl_comm, double* G, int64_t g_stride, int64_t pa,
                                  int n_blocks, double* buf, void* stream) {
    if (!ctx || !G || !buf) return fail(ctx, 1, "slm_gram_allreduce: null argument");
    if (n_blocks < 1 || n_blocks > SLM_MAX_FOLDS) return fail(ctx, 1, "slm_gram_allreduce: n_blocks out of range");
    if (int rc = slm_tri_pack(ctx, G, g_stride, pa, n_blocks, buf, stream)) return rc;
    if (nccl_comm)  // NULL: single rank, the complement alone
        if (int rc = slm_allreduce_sum(ctx, nccl_comm, buf, (int64_t)n_blocks * slm_tri_size(pa), stream)) return rc;
    return slm_tri_complement(ctx, buf, pa, n_blocks, G, g_stride, stream);
}

