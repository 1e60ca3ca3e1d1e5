/*
 * sparselm_b200 -- C ABI of the B200 solver engine for sparse-lm's convex estimators.
 *
 * This is the drop-in boundary for the reference's solve seam
 *     CVXRegressor._solve(X, y, solver_options)      src/sparselm/model/_base.py:512-519
 * (overrides: model/_lasso.py:486-502, model/_adaptive_lasso.py:206-232, 515-524)
 * and for the (candidate x fold) fan-out that drives it
 *     GridSearchCV.fit / evaluate_candidates          src/sparselm/model_selection.py:291-359
 * The reference is pure Python; a maintainer binds this library with ctypes
 * (see INTEGRATION.md).  All pointers named *_dev are device pointers owned by the
 * caller (the Python host allocates them as torch tensors); the engine never
 * frees caller memory.  Every call is ordered on the given CUDA stream
 * (a cudaStream_t passed as void*).  Return value 0 = success; otherwise an
 * error code and slm_last_error() describes it.  No C++ exception crosses
 * this boundary.
 *
 * Layouts.  The design matrix lives on the device as the *augmented* row-major
 * matrix Xa[n][lda] = [ X | y | 1 | 0-pad ], lda = slm_padded_cols(p).  One
 * symmetric Gram of Xa (pa x pa, pa == lda) therefore carries X^T X, X^T y,
 * y^T y, the column sums and n.  Batched solver state is feature-major:
 * Z[f][j][k], fold f, feature j, grid column k (k contiguous, row stride ldz,
 * ldz % 8 == 0), so one fold's coefficient batch is the row-major B operand of
 * the tensor-core Gram apply.
 */
#ifndef SPARSELM_B200_H
#define SPARSELM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLM_MAX_FOLDS 16

typedef struct slm_ctx slm_ctx;

/* ---- lifecycle ----------------------------------------------------------- */
int slm_version(void);
int slm_create(int device, slm_ctx** out);
void slm_destroy(slm_ctx* ctx);
/* engine switches (the SLM_* environment variables read at slm_create, settable later):
 * "coop" (cooperative few-column iterations),
 * "tma" (bit mask of the kernel families fed by TMA + mbarrier instead of cp.async: 1 Gram build,
 * 2 dense Gram apply, 4 row-sparse Gram apply, 8 / 16 wide padded-pitch bands instead of 128-byte
 * swizzled boxes for the gather / tiled kernels; default 15), "fused_prox" (default 1: one prox_fused_kernel per
 * iteration on the iterate buffers, the Gram applied to the iterate itself; 0: the two-kernel iteration on a
 * materialised extrapolated point), "force_apply_shape" / "force_sparse_shape" /
 * "force_syrk_shape" (tile menu overrides of tools/gemm_probe.py, -1 = automatic). */
int slm_set_option(slm_ctx* ctx, const char* name, int value);
const char* slm_last_error(const slm_ctx* ctx);
int slm_sm_count(const slm_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t slm_launch_count(const slm_ctx* ctx);
/* how many of those were TMA-fed GEMM launches (gemm_f64_tma_kernel) */
int64_t slm_tma_launch_count(const slm_ctx* ctx);
/* average device time in ms of the `which` kernel family since the last reset,
 * measured with CUDA events on the launching stream when timing is enabled.
 * which: 0 = gram build, 1 = gram apply (solver), 2 = prox, 3 = gap, 4 = score,
 *        5 = gram apply inside the Lipschitz power iteration */
int slm_timing_enable(slm_ctx* ctx, int on);
int slm_timing_read(slm_ctx* ctx, int which, double* total_ms, int64_t* launches, double* flops);
int slm_timing_reset(slm_ctx* ctx);

/* pa = lda = round_up(p + 2, 8) */
int64_t slm_padded_cols(int64_t p);

/* ---- K1: design packing and Gram build ----------------------------------- */
/* replaces: X, y arrival in CVXRegressor.fit / _preprocess_data (_base.py:173-227).
 * Xa[r][0:p] = sqrt(sw_r) * X[perm? no: r][col_perm[j]], Xa[r][p] = sqrt(sw_r) y_r,
 * Xa[r][p+1] = sqrt(sw_r), rest 0.  col_perm_dev (int32[p]) may be NULL (identity);
 * row_perm_dev (int64[n]) may be NULL; sw_dev may be NULL. */
int slm_pack_design(slm_ctx* ctx, const double* X_dev, int64_t ldx, const double* y_dev,
                    const double* sw_dev, const int32_t* col_perm_dev,
                    const int64_t* row_perm_dev, int64_t n, int64_t p, double* Xa_dev,
                    int64_t lda, void* stream);

/* Gblk[f] = Xa[rows_f]^T Xa[rows_f], rows_f = [row_ptr[f], row_ptr[f+1]); FP64 DMMA
 * SYRK (upper tiles + mirror).  replaces: the data term cp.sum_squares(X @ beta - y)
 * (_lasso.py:120) being re-canonicalised for every fit.  row_ptr is a HOST array. */
int slm_gram_blocks(slm_ctx* ctx, const double* Xa_dev, int64_t lda, const int64_t* row_ptr,
                    int n_blocks, double* Gblk_dev, void* stream);
/* G += Xa[r0:r1]^T Xa[r0:r1] (same kernel, the first writer of every tile adds to what G holds,
 * upper tiles and their mirror alike): lets the Gram of a host-resident design be accumulated
 * block of rows by block of rows while the next block is still on the PCIe bus. */
int slm_gram_block_add(slm_ctx* ctx, const double* Xa_dev, int64_t lda, int64_t r0, int64_t r1,
                       double* G_dev, void* stream);

/* Gram of an arbitrary row set, for n_problems problems at once (CV splits that are not one partition of the
 * rows): G[s] (+|-)= Xa[idx_s]^T Xa[idx_s], FP64 DMMA, upper tiles + mirror.  Xa_dev is [n][lda]; the row lists
 * are rows_dev[row_ptr[s] .. row_ptr[s+1]) (device int32, ascending; row_ptr is a HOST array of n_problems + 1
 * offsets); Gram s is at G_dev + s * g_stride.  accumulate == 0: G[s] is overwritten; != 0: the product is added
 * to what G[s] holds (as slm_gram_block_add).  negate != 0: the product enters with a minus sign (with
 * accumulate: a downdate G[s] -= Xa[idx]^T Xa[idx]).  An empty list leaves G[s] untouched.  Bit-reproducible. */
int slm_gram_rows_update(slm_ctx* ctx, const double* Xa_dev, int64_t n, int64_t lda, int n_problems,
                         const int64_t* row_ptr, const int32_t* rows_dev, double* G_dev, int64_t g_stride,
                         int accumulate, int negate, void* stream);

/* in place: Gtot = sum_f Gblk[f]; Gblk[f] <- Gtot - Gblk[f]  (training Gram of fold f
 * when the blocks are the CV test folds, model_selection.py:304-323). */
int slm_gram_complement(slm_ctx* ctx, double* Gblk_dev, int n_blocks, int64_t pa,
                        double* Gtot_dev, void* stream);

/* Row-sharded build (SURVEY 8e): every rank builds the Gram blocks of its own rows and the
 * blocks are summed over the ranks with one NCCL all-reduce.  A Gram is symmetric, so only its
 * upper triangle travels: slm_tri_pack copies n_grams Grams (stride g_stride doubles) into
 * buf_dev[n_grams][slm_tri_size(pa)] (row i = columns i..pa-1), slm_tri_unpack restores the full
 * matrices (upper part + mirror) from the reduced buffer. */
int64_t slm_tri_size(int64_t pa);
int slm_tri_pack(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int n_grams,
                 double* buf_dev, void* stream);
int slm_tri_unpack(slm_ctx* ctx, const double* buf_dev, int64_t pa, int n_grams, double* G_dev,
                   int64_t g_stride, void* stream);

/* slm_tri_complement: the reduced packed buffer buf_dev[n_blocks][slm_tri_size(pa)] -> the n_blocks
 * training Grams (sum of the other blocks) followed by the total in G_dev[n_blocks + 1][pa][pa] (full
 * symmetric matrices): slm_tri_unpack + slm_gram_complement in one pass.
 *
 * Collectives of the sharded search on the CALLER's NCCL communicator (an ncclComm_t passed as void*; the
 * reference side gets it from its process group, e.g. torch.distributed's ProcessGroupNCCL._comm_ptr()).
 * The library does not link NCCL: it uses the NCCL already loaded in the process, so communicator and
 * entry points match.  All are enqueued on `stream`; NCCL's usual rule applies (every rank issues the same
 * collectives in the same order).
 *   slm_gram_allreduce: this rank's partial fold blocks G_dev[n_blocks][pa][pa] -> training Grams + total
 *       of all ranks in G_dev[n_blocks + 1][pa][pa] (pack upper triangles, ONE ncclAllReduce, unpack +
 *       complement); buf_dev holds n_blocks * slm_tri_size(pa) doubles; nccl_comm NULL = single rank.
 *   slm_allreduce_sum: in-place sum of count doubles (the zero-padded CV score / info tables).
 *   slm_gather_results: ncclAllGather of count_per_rank doubles per rank (coefficients + intercepts of the
 *       columns a rank solved) so that every rank can score its rows of every test fold. */
int slm_tri_complement(slm_ctx* ctx, const double* buf_dev, int64_t pa, int n_blocks, double* G_dev,
                       int64_t g_stride, void* stream);
int slm_gram_allreduce(slm_ctx* ctx, void* nccl_comm, double* G_dev, int64_t g_stride, int64_t pa,
                       int n_blocks, double* buf_dev, void* stream);
int slm_allreduce_sum(slm_ctx* ctx, void* nccl_comm, double* buf_dev, int64_t count, void* stream);
int slm_gather_results(slm_ctx* ctx, void* nccl_comm, const double* send_dev, double* recv_dev,
                       int64_t count_per_rank, void* stream);

/* Diagnostic of the TMA path (gemm_f64_tma.cuh): loads the [16 rows][16 doubles] box at (row0, col0) of
 * the row-major device matrix A_dev[rows][ld] with a tiled tensor map and the four rows r[0..3] at col0
 * with a tile::gather4 map (both 128-byte swizzled) and writes the raw shared-memory images to
 * out_dev[320] (256 + 64 doubles).  tests/test_gpu_tma.py checks them against the layout the
 * consumers assume (chunk XOR (row & 7), zero fill outside the matrix). */
int slm_tma_probe(slm_ctx* ctx, const double* A_dev, int64_t rows, int64_t ld, int32_t col0, int32_t row0,
                  const int32_t* r4_host, double* out_dev, void* stream);

/* in-place centering of one augmented Gram using its ones row/column
 * (fit_intercept=True, _base.py:216-222): G <- G - s s^T / n on the [0,p] block. */
int slm_gram_center(slm_ctx* ctx, double* G_dev, int64_t pa, int64_t p, void* stream);

/* G_ext[a][b] = G[idx[a]][idx[b]] for a,b < pe; rows/cols pe, pe+1 (y, ones) follow.
 * replaces X_ext = X[:, beta_indices] (_lasso.py:461). pae = slm_padded_cols(pe). */
int slm_gram_gather(slm_ctx* ctx, const double* G_dev, int64_t pa, int64_t p,
                    const int32_t* idx_dev, int64_t pe, double* Gext_dev, int64_t pae,
                    void* stream);

/* lambda_max(G[0:p,0:p]) for n_grams Grams (stride g_stride doubles) by batched block
 * power iteration on the tensor-core apply; result (HOST array lam[n_grams]) is the
 * largest Rayleigh quotient seen (a lower bound; callers add a margin).
 * work_dev: >= slm_lipschitz_workspace(p, n_grams) bytes. */
size_t slm_lipschitz_workspace(int64_t p, int n_grams);
/* same, result left on the device (lam_dev[n_grams]) and NO host synchronisation: the step
 * sizes then reach slm_solve_batch through slm_batch.lipschitz_dev */
int slm_lipschitz_dev(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int64_t p,
                      int n_grams, int iters, void* work_dev, double* lam_dev, void* stream);
int slm_lipschitz(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int64_t p,
                  int n_grams, int iters, void* work_dev, double* lam_host, void* stream);

/* ---- K5-K7: the batched accelerated proximal-gradient solve --------------- */
typedef struct slm_batch {
    /* problem data */
    int32_t n_folds;     /* number of Grams in this batch (<= SLM_MAX_FOLDS)          */
    int32_t n_groups;    /* number of penalty groups (groups contiguous in feature order) */
    int64_t p;           /* features                                                   */
    int64_t pa;          /* leading dimension of every Gram                            */
    int64_t ldz;         /* row stride of all [p][ldz] / [G][ldz] arrays (mult. of 8)  */
    const double* G_dev; /* Gram f at G_dev + f*g_stride; c_f is its row p, yty = [p][p] */
    int64_t g_stride;
    const int32_t* gptr_dev; /* int32[n_groups+1]; NULL => every feature its own group */
    int32_t K[SLM_MAX_FOLDS];        /* grid columns of fold f (<= ldz)               */
    double n_obs[SLM_MAX_FOLDS];     /* n of the data term 1/(2n)                      */
    double lipschitz[SLM_MAX_FOLDS]; /* L >= lambda_max(G_f)/n_f                       */
    /* penalty weights, all [F][rows][ldz] device arrays with fold stride rows*ldz    */
    const double* lam1_dev; /* [F][ldz] l1 weight per column, used when W1_dev == NULL */
    const double* W1_dev;   /* [F][p][ldz] per-coefficient l1 weights or NULL          */
    const double* W2_dev;   /* [F][n_groups][ldz] group-l2 weights or NULL (=0)        */
    const double* D2_dev;   /* [F][n_groups][ldz] ridge weights or NULL (=0)           */
    /* state: B in = start point, out = solution                                       */
    double* B_dev;          /* [F][p][ldz]                                             */
    const int32_t* skip_dev; /* [F][ldz] or NULL: columns with skip != 0 are left untouched
                              * (adaptive chains whose weights already converged)       */
    void* work_dev;         /* >= slm_solve_workspace(...) bytes                        */
    size_t work_bytes;
    /* control */
    double tol;        /* stop when gap <= tol * max(|primal|, floor_rel * yty/(2n))    */
    double floor_rel;
    int32_t max_iter;
    int32_t check_every;
    /* per-column results, [F][ldz] device arrays (may be NULL) */
    double* gap_dev;
    double* primal_dev;
    int32_t* n_iter_dev;
    int32_t* status_dev; /* 0 converged, 1 max_iter reached, 2 non-finite */
    const double* lipschitz_dev; /* [n_folds] device array of L, or NULL; overrides lipschitz[]
                                  * (lets the Lipschitz estimate feed the solve with no host sync) */
    /* host outputs */
    int32_t iters_run;     /* outer iterations executed */
    int32_t n_unconverged; /* columns that hit max_iter */
    int32_t max_group;     /* in: rows of the largest group (gptr_dev given), 0 = unknown; lets the
                              few-column cooperative iterations size their row ranges */
} slm_batch;

size_t slm_solve_workspace(int64_t p, int64_t ldz, int n_folds, int n_groups);

/* replaces cp.Problem.solve for every (fold, grid column) at once (_base.py:516). */
int slm_solve_batch(slm_ctx* ctx, slm_batch* batch, void* stream);

/* ---- K8: adaptive reweighting (_adaptive_lasso.py:196-204, 364-374, 712-726) -----
 * W1[j][k] = a1[k] * alpha[k] / (|B[j][k]| + eps)            (if W1_dev != NULL)
 * W2[g][k] = a2[k] * gw[g] * alpha[k] / (||B_g[:,k]|| + eps)  (if W2_dev != NULL)
 * dnorm[k] = || [W2;W1]_new - [W2;W1]_old ||_2  (convergence test :189-194, :698-710) */
int slm_adaptive_update(slm_ctx* ctx, const double* B_dev, int64_t p, int64_t ldz, int32_t K,
                        int32_t n_groups, const int32_t* gptr_dev, const double* gw_dev,
                        const double* a1_dev, const double* a2_dev, const double* alpha_dev,
                        double eps, double* W1_dev, double* W2_dev, double* dnorm_dev,
                        void* stream);

/* ---- K9: overlap fold-back (_lasso.py:492-501) ----------------------------------
 * coef[j][k] = sum_{t in [inv_ptr[j], inv_ptr[j+1])} Bext[inv_idx[t]][k]
 * (CSR inverse of beta_indices, summed in ascending order: deterministic). */
int slm_fold_back(slm_ctx* ctx, const double* Bext_dev, const int32_t* inv_ptr_dev,
                  const int32_t* inv_idx_dev, int64_t p, int64_t ldz, int32_t K,
                  double* coef_dev, void* stream);

/* ---- K10: CV scoring (sklearn scorer inside _fit_and_score, model_selection.py:305)
 * rows [r0, r1) of Xa are the test fold; B [p][ldz]; intercept[k] may be NULL.
 * out_dev[0][k] = sum (y - yhat)^2, out_dev[1][k] = sum |y - yhat|  (ldz stride).
 * rows_scaled != 0: the rows were packed with sample weights (sqrt(sw_i) [x_i, y_i, 1]) and the
 * scorer is unweighted, as sklearn's is for fit_params (model_selection.py:266): residuals are
 * divided by the row's sqrt(sw_i) column (all weights must be > 0).
 * yhat_dev: scratch [(r1-r0) + 256][ldz] (predictions, then partial sums). */
int slm_cv_score(slm_ctx* ctx, const double* Xa_dev, int64_t lda, int64_t p, int64_t r0,
                 int64_t r1, const double* B_dev, int64_t ldz, int32_t K,
                 const double* intercept_dev, int32_t rows_scaled, double* yhat_dev,
                 double* out_dev, void* stream);

/* n scoring problems in one tensor-core launch (row-sharded scoring of a sharded grid: this rank's slice of
 * every fold's rows x the columns each rank solved on that fold).  All arrays are HOST arrays of length n;
 * B[i] / intercept[i] / yhat[i] / out[i] are device pointers.  Problem i scores rows [r0[i], r1[i]) of Xa
 * against the K[i] columns of B[i] ([p][ldb[i]], ldb even, B[i] 16-byte aligned); yhat[i] is scratch
 * [(r1-r0) + 256][ldy[i]] (ldy a multiple of 8, >= K[i] rounded up to 8); out[i] is [2][ldy[i]] as in
 * slm_cv_score.  intercept may be NULL (no intercepts at all) or hold NULL entries. */
int slm_cv_score_many(slm_ctx* ctx, const double* Xa_dev, int64_t lda, int64_t p, int32_t n,
                      const int64_t* r0, const int64_t* r1, const double* const* B_dev, const int64_t* ldb,
                      const int32_t* K, const double* const* intercept_dev, int32_t rows_scaled,
                      double* const* yhat_dev, const int64_t* ldy, double* const* out_dev, void* stream);

/* slm_cv_score_many with a row list per problem instead of a row range: problem i scores the n_rows[i] rows
 * rows_dev[i][0 .. n_rows[i]) of Xa (device int32 array; rows_dev[i] is a device pointer, the other arrays are
 * HOST arrays of length n as in slm_cv_score_many).  yhat[i] is scratch [n_rows[i] + 256][ldy[i]]. */
int slm_cv_score_rows(slm_ctx* ctx, const double* Xa_dev, int64_t lda, int64_t p, int32_t n,
                      const int32_t* const* rows_dev, const int64_t* n_rows, const double* const* B_dev,
                      const int64_t* ldb, const int32_t* K, const double* const* intercept_dev, int32_t rows_scaled,
                      double* const* yhat_dev, const int64_t* ldy, double* const* out_dev, void* stream);

/* Residual statistics beyond the two sums, for the CV scorers that need them (neg_max_error,
 * neg_mean_absolute_percentage_error, neg_median_absolute_error).  rows_dev == NULL: problem i is the row range
 * [r0[i], r1[i]) as in slm_cv_score_many; else the row list rows_dev[i] of n_rows[i] rows as in slm_cv_score_rows
 * (r0 / r1 may then be NULL, and n_rows may be NULL with ranges).  out[i] is [5][ldy[i]]:
 *   row 0: sum r^2, row 1: sum |r| (bitwise what slm_cv_score_many / slm_cv_score_rows return),
 *   row 2: max |r|                        (SLM_STAT_MAX),
 *   row 3: sum |r| / max(|y|, DBL_EPSILON) (SLM_STAT_MAPE; y recovered like r when rows_scaled),
 *   row 4: median |r|                     (SLM_STAT_MEDIAN; the mean of the two middle values when the count is
 *                                          even, as numpy.median).
 * r is the residual of the sums (divided by the row's sqrt(sw) column when rows_scaled).  Rows 2-4 are written
 * only when their bit of `stats` is set; stats == 0 is slm_cv_score_many / slm_cv_score_rows.  With stats != 0,
 * rows [0, m) of yhat[i] hold the residuals that were reduced when the call's work completes.  max and median are
 * exact (the median is a radix select on the bit patterns, no arithmetic but the final (a + b) / 2; a NaN residual
 * makes both NaN); the percentage sum uses the fixed two-stage order of the sums: every result is bit-reproducible.
 * yhat[i] is scratch [m + 256][ldy[i]] as in slm_cv_score_many. */
#define SLM_STAT_MAX (1 << 2)
#define SLM_STAT_MAPE (1 << 3)
#define SLM_STAT_MEDIAN (1 << 4)
int slm_cv_score_stats(slm_ctx* ctx, const double* Xa_dev, int64_t lda, int64_t p, int32_t n,
                       const int64_t* r0, const int64_t* r1, const int32_t* const* rows_dev, const int64_t* n_rows,
                       const double* const* B_dev, const int64_t* ldb, const int32_t* K,
                       const double* const* intercept_dev, int32_t rows_scaled, int32_t stats,
                       double* const* yhat_dev, const int64_t* ldy, double* const* out_dev, void* stream);

/* ---- K11: stability selection counts (DESIGN section 2 item 17) ------------------------------------
 * coef_dev is the [F][p][ldz] coefficient table of F fits x K candidate columns (slm_solve_batch / fold-back
 * layout, F <= SLM_MAX_FOLDS, K <= ldz).  Coefficient j of fit (f, k) is selected iff
 *   |coef[f][j][k]| > rel_tol * max_j' |coef[f][j'][k]|
 * (an all-zero fit selects nothing; a NaN coefficient is never selected; columns k >= K are never read).
 *   counts_dev[j][k] += number of fits f of the call that select j for candidate k   (int32 [p][K])
 *   union_dev[f][j]   = 1 if some candidate k < K of fit f selects j, else left as is  (uint8 [F][p])
 * Both accumulate over calls; no atomics on the counts, so the results are deterministic.  Only enqueues work. */
int slm_support_counts(slm_ctx* ctx, const double* coef_dev, int F, int64_t p, int64_t ldz, int K, double rel_tol,
                       int32_t* counts_dev, uint8_t* union_dev, void* stream);

/* intercept[k] = ybar - mu^T B[:,k] from the (uncentred) training Gram's ones row
 * (LinearModel._set_intercept, _base.py:202). */
int slm_intercepts(slm_ctx* ctx, const double* G_dev, int64_t pa, int64_t p,
                   const double* B_dev, int64_t ldz, int32_t K, double* intercept_dev,
                   void* stream);

/* Second-order phase of the batched solve (pure group penalties; slm_newton_step_l1 below adds the l1 term;
 * DESIGN section 2 item 13): ONE
 * lock-step damped Newton step on the active groups of k columns, in this library's kernels --
 * Hessian assembly from the Gram, batched blocked Cholesky (trailing updates on the tensor-core
 * GEMM), blocked triangular solves, Armijo line search on objective differences.
 * Column c works on Gram fold_host[c] with nobs_dev[c] rows; X_dev [k][ldv] (ldv = round_up(p, 8))
 * holds its point in solver feature order and is updated in place when a step is accepted;
 * W2_dev / D2_dev [k][n_groups] are its group and ridge weights (D2_dev may be NULL); gptr_dev
 * [n_groups+1], gid_dev [p] describe the groups.  out_dev [k][4] = {accepted, step length,
 * Newton decrement -grad'd, factorisation failed}.  Only enqueues work on the stream. */
size_t slm_newton_workspace(int64_t p, int32_t n_groups, int32_t k, int n_folds);
int slm_newton_step(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                    int32_t k, const int32_t* fold_host, const double* nobs_dev, double* X_dev,
                    const double* W2_dev, const double* D2_dev, const int32_t* gptr_dev, const int32_t* gid_dev,
                    int32_t n_groups, void* work_dev, size_t work_bytes, double* out_dev, void* stream);

/* The same step for penalties with an l1 term (Lasso, SparseGroupLasso and their adaptive variants):
 * W1_dev [k][ldv] holds every column's per-coordinate l1 weights in solver feature order (NULL: pure group
 * penalty, bitwise the same as slm_newton_step).  On the manifold of fixed signs a coordinate is active iff it
 * is non-zero; the line search starts from min(1, t_cross), t_cross the first step length at which a
 * coordinate changes sign, and a step accepted at t_cross stores the coordinates that reach zero as exact
 * zeros (out_dev[c][1] reports the step taken).  Without a group structure pass one group of all p
 * coordinates with zero weight.  Same workspace as slm_newton_step. */
int slm_newton_step_l1(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int64_t p, int n_folds,
                       int32_t k, const int32_t* fold_host, const double* nobs_dev, double* X_dev,
                       const double* W2_dev, const double* D2_dev, const double* W1_dev, const int32_t* gptr_dev,
                       const int32_t* gid_dev, int32_t n_groups, void* work_dev, size_t work_bytes, double* out_dev,
                       void* stream);

/* Unpenalised least squares on a Gram (OrdinaryLeastSquares, reference model/_ols.py:57-65:
 * argmin 1/(2n) ||X b - y||^2): conjugate gradients on G b = c, c = row p of the Gram, every
 * product G d through the tensor-core apply.  From b = 0 the iterates stay in range(G), so a
 * rank-deficient (p > n) consistent system converges to its minimum-norm solution.  Stops on
 * ||c - G b|| <= tol ||c|| (checked against the recomputed residual) or after max_iter products.
 * X8_dev: [p][8] out, the solution is column 0 (stride 8: the layout slm_intercepts and
 * slm_cv_score take with ldz = 8).  iters_host / relres_host may be NULL.  Synchronises.
 * shift_dev (may be NULL): p non-negative numbers added to the diagonal of G -- the ridge
 * n * delta_g(j) of a penalised estimator called with alpha = 0 (valid in the reference,
 * _lasso.py:77-79: the interval is closed at 0), whose columns the host routes here because the
 * duality-gap test of the proximal iterations degenerates without a penalty. */
size_t slm_gram_cg_workspace(int64_t p);
int slm_gram_cg(slm_ctx* ctx, const double* G_dev, int64_t pa, int64_t p, const double* shift_dev,
                double tol, int32_t max_iter, void* work_dev, size_t work_bytes, double* X8_dev,
                int32_t* iters_host, double* relres_host, void* stream);

/* plain batched tensor-core apply GZ_f = G_f Z_f (exposed for tests / roofline runs) */
int slm_gram_apply(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa, int64_t p,
                   int n_folds, const int32_t* K, const double* Z_dev, int64_t ldz,
                   double* GZ_dev, void* stream);

/* Row-sparse form of the same apply, as the solver uses it: the iterates of a sparse
 * linear model are mostly exact zeros, so for every chunk of chunk_w grid columns only
 * the rows j of Z_f with a non-zero in the chunk (and, by symmetry, the matching rows of
 * G_f) enter the contraction.  The row lists are built on the device and the kernel
 * partitions its stream-K work from the device-side counts.  Same result as
 * slm_gram_apply up to summation order.  work_dev: slm_rowsparse_workspace bytes. */
size_t slm_rowsparse_workspace(int64_t p, int64_t ldz, int n_folds);
int slm_gram_apply_rowsparse(slm_ctx* ctx, const double* G_dev, int64_t g_stride, int64_t pa,
                             int64_t p, int n_folds, const int32_t* K, const double* Z_dev,
                             int64_t ldz, double* GZ_dev, int chunk_w, void* work_dev,
                             size_t work_bytes, void* stream);

/* flops of the solver's Gram applies since the last slm_timing_reset: executed (rows of the
 * support lists x real columns x 2p) and dense-equivalent (2 p^2 K_active). */
int slm_apply_stats(slm_ctx* ctx, double* executed_flops, double* dense_flops);

/* ---- standardize=True (reference _lasso.py:249-252; ridged variant :776-789) ----------
 * The reference penalises ||X_g b_g||_2, resp. ||sqrtm(X_g^T X_g + sqrt(delta_g) I) b_g||_2,
 * instead of ||b_g||_2.  With A_g = G_gg (+ shift_g I) = R_g^T R_g (Cholesky) both are
 * ||R_g b_g||, so in gamma_g = R_g b_g the problem is a plain group Lasso on the Gram
 * W^T G W, W = blockdiag(W_g), W_g = R_g^{-1}.
 *
 * slm_group_whiten_factors: W_g for every group of ONE Gram, stored m_g x m_g row-major at
 *   W_dev + wptr[g] (wptr_dev: int64[n_groups+1], wptr[g+1]-wptr[g] = m_g^2); scratch_dev has
 *   the size of W_dev; shift_dev[n_groups] (sqrt(delta_g)) may be NULL; info_dev[0] is
 *   incremented for every group whose block is not numerically positive definite (the
 *   group's columns are then linearly dependent on the training rows).
 * slm_gram_whiten: Gout = W^T G W on the feature block; the y / ones rows and columns are
 *   transformed on one side, so c = X^T y becomes W^T c and y^T y is kept.  ridge_dev[n_groups]
 *   (delta_g, may be NULL) folds the ridge 1/2 delta_g ||b_g||^2 into the Gram:
 *   Gout_gg += ridge_scale * delta_g * W_g^T W_g with ridge_scale = n of the data term.
 *   tmp_dev: pa*pa doubles.  G, tmp, Gout distinct.
 * slm_coef_unwhiten: B[g rows][k] = W_g Bg[g rows][k] (coefficients back in the caller's
 *   variables) for K columns of a [p][ldz] array. */
int slm_group_whiten_factors(slm_ctx* ctx, const double* G_dev, int64_t pa, int64_t p,
                             const int32_t* gptr_dev, const int64_t* wptr_dev, int32_t n_groups,
                             const double* shift_dev, double* W_dev, double* scratch_dev,
                             int32_t* info_dev, void* stream);
int slm_gram_whiten(slm_ctx* ctx, const double* G_dev, int64_t pa, int64_t p,
                    const int32_t* gptr_dev, const int64_t* wptr_dev, int32_t n_groups,
                    const double* W_dev, const double* ridge_dev, double ridge_scale,
                    double* tmp_dev, double* Gout_dev, void* stream);
int slm_coef_unwhiten(slm_ctx* ctx, const double* Bg_dev, int64_t p, int64_t ldz, int32_t K,
                      const int32_t* gptr_dev, const int64_t* wptr_dev, int32_t n_groups,
                      const double* W_dev, double* B_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPARSELM_B200_H */
