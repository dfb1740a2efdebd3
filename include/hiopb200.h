/* hiopb200.h -- C-ABI of the B200-native (sm_100a) engine for HiOp's KKT assemble + factor + solve hot path.
 *
 * Drop-in boundary: every entry point below replaces one reference interface (cited as file:line relative to
 * the LLNL/hiop tree). The library is libhiopb200.so; INTEGRATION.md shows the C++ adapter classes
 * (hiopLinSolverSymDenseB200, hiopKKTLinSysLowRankB200, hiopHessianLowRankB200) a HiOp maintainer would add on top.
 *
 * Conventions (copied from the reference's own C interface, src/Interface/hiopInterface.h): plain pointers and
 * sizes, `int` status returns (HB_OK = 0, negative = error; hb_last_error() gives the text), no exceptions cross the
 * boundary, opaque handles owned by the engine, inputs owned by the caller.
 *   - All `double*` / `int*` arguments are DEVICE pointers unless the function name ends in `_host` or the
 *     parameter is documented as host.
 *   - All arithmetic is IEEE FP64; patterns ("select" vectors) are FP64 0.0/1.0 as in the reference
 *     (src/LinAlg/hiopVectorPar.cpp:782).
 *   - Dense matrices are row-major like hiopMatrixDenseRowMajor (src/LinAlg/hiopMatrixDenseRowMajor.cpp:86-96).
 *   - Element counts / offsets are 64-bit (`long long`); the reference's `int` indexing cannot address the n=4e6,
 *     m=4000 configuration.
 *   - Every context owns one CUDA stream; calls are asynchronous on that stream unless they return a host scalar.
 *   - There is no CPU fallback anywhere: without a CUDA device hb_ctx_create fails with HB_ERR_CUDA.
 */
#ifndef HIOPB200_H
#define HIOPB200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_OK 0
#define HB_ERR_INVALID (-1)   /* bad argument */
#define HB_ERR_CUDA (-2)      /* CUDA runtime error (message in hb_last_error) */
#define HB_ERR_ALLOC (-3)     /* device allocation failed */
#define HB_ERR_NUMERIC (-4)   /* factorization broke down (not SPD / zero pivot) */
#define HB_ERR_STATE (-5)     /* call order violated (e.g. solve before condense) */
#define HB_ERR_COMM (-6)      /* NCCL not available / communicator error */

typedef struct hb_ctx hb_ctx;
typedef struct hb_lowrank hb_lowrank;
typedef struct hb_symdense hb_symdense;
typedef struct hb_mds hb_mds;

/* ------------------------------------------------------------------------------------------------------------
 * Context, memory, streams
 * ------------------------------------------------------------------------------------------------------------ */
const char* hb_version(void);
const char* hb_last_error(void);
/* number of kernel launches issued by this library since load (all contexts); feeds bench.py's gpu_launches */
long long hb_launch_count(void);

/* Replaces the ExecSpace/MemBackend plumbing (src/ExecBackends/) for this path: one device, one stream. */
int hb_ctx_create(int device, hb_ctx** out);
int hb_ctx_destroy(hb_ctx* ctx);
int hb_ctx_sync(hb_ctx* ctx);
/* the cudaStream_t of the context (so a host framework can order its own work/events against it) */
void* hb_ctx_stream(hb_ctx* ctx);
int hb_ctx_device(hb_ctx* ctx);

/* Kernel-level timing for roofline reporting: when enabled, CUDA events bracket the dominant kernel of the condensation -- whichever
 * ran: the FP64 DMMA SYRK (k_syrk_ws) or the int8-slice tcgen05 GEMM (k_oz_gemm; with column chunks, the slicing and GEMMs of all
 * chunks) -- on the context stream; hb_ctx_last_syrk_ms waits for it and returns its device duration. */
int hb_ctx_enable_timing(hb_ctx* ctx, int on);
/* Per-phase timeline of one quasi-Newton step (per-rank evidence for the multi-GPU runs): hb_ctx_phase_timeline(ctx, 1, NULL) arms the
 * marks, the next hb_lowrank_update + condense + solve_compressed records an event after each phase, hb_ctx_phase_timeline(ctx, 0, ms)
 * returns 12 durations in ms: update, row maxima (+ fused row dots), slicing, GEMM + fix-up (the whole condensation with the FP64 kernel),
 * all-reduce, V/U/N assembly, Cholesky, H^-1 rx, J dx (+ all-reduce), SPD solve, J^T dy, H^-1 rx (second). With an int8-slice
 * condensation in several column chunks (hb_lowrank_last_condense_chunks > 1) the slicing entry is 0 and the GEMM entry holds the
 * slicing and GEMM of every chunk. */
int hb_ctx_phase_timeline(hb_ctx* ctx, int on, float* ms_host10);
int hb_ctx_last_syrk_ms(hb_ctx* ctx, float* ms_host);

/* Measured roofline denominators of this device (a few milliseconds each, CUDA events on the context stream):
 * which = 0: FP64 tensor pipe, mma.sync.m8n8k4.f64 issued back to back from registers (TFLOP/s);
 * which = 1: tcgen05.mma.kind::i8 M=128 N=256 K=32 issued back to back on resident operands (TOP/s, 2 ops per MAC). */
int hb_microbench_peak(hb_ctx* ctx, int which, double* result_host);

int hb_malloc(hb_ctx* ctx, size_t bytes, void** dptr);
int hb_free(hb_ctx* ctx, void* dptr);
int hb_malloc_host(hb_ctx* ctx, size_t bytes, void** hptr); /* pinned */
int hb_free_host(hb_ctx* ctx, void* hptr);
int hb_memcpy_h2d(hb_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes); /* async on the ctx stream */
int hb_memcpy_d2h(hb_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes); /* async on the ctx stream */
int hb_memcpy_d2d(hb_ctx* ctx, void* dst_dev, const void* src_dev, size_t bytes);
int hb_memset(hb_ctx* ctx, void* dst_dev, int byte, size_t bytes);

/* Multi-GPU: column (n) partition exactly like the reference's MPI layout (src/Optimization/hiopHessianLowRank.hpp:88-89).
 * The 128-byte NCCL unique id is created on rank 0 (hb_comm_unique_id) and broadcast by the host program.
 * After hb_comm_init every reduction the reference does with MPI_Allreduce on this path
 * (src/Optimization/hiopHessianLowRank.cpp:459,590,591; src/LinAlg/hiopMatrixDenseRowMajor.cpp:487;
 * src/LinAlg/hiopVectorPar.cpp:474-548) is done with ncclAllReduce on the context stream. */
int hb_comm_unique_id(void* id128_host);
int hb_comm_init(hb_ctx* ctx, int nranks, int rank, const void* id128_host);
int hb_comm_size(hb_ctx* ctx);
int hb_comm_rank(hb_ctx* ctx);
/* in-place sum all-reduce of `count` doubles on the context stream (no-op for a single rank) */
int hb_allreduce_sum(hb_ctx* ctx, double* buf_dev, long long count);

/* ------------------------------------------------------------------------------------------------------------
 * hiopVector elementwise ops + reductions (B3; src/LinAlg/hiopVector.hpp:62-1017, oracle: hiopVectorPar.cpp)
 * One launch each; 128-bit vectorised, grid-stride over 148 x k CTAs.
 * ------------------------------------------------------------------------------------------------------------ */
int hb_vec_set(hb_ctx*, long long n, double* y, double c);                                  /* setToConstant */
int hb_vec_copy(hb_ctx*, long long n, double* y, const double* x);                          /* copyFrom */
int hb_vec_scale(hb_ctx*, long long n, double* y, double alpha);                            /* scale        :657 */
int hb_vec_axpy(hb_ctx*, long long n, double* y, double alpha, const double* x);            /* axpy         :662-670 */
int hb_vec_axzpy(hb_ctx*, long long n, double* y, double alpha, const double* x, const double* z);   /* :710-734 */
int hb_vec_axdzpy(hb_ctx*, long long n, double* y, double alpha, const double* x, const double* z);  /* :736-765 */
int hb_vec_axdzpy_w_pattern(hb_ctx*, long long n, double* y, double alpha, const double* x, const double* z,
                            const double* select);                                          /* :767-790 */
int hb_vec_component_mult(hb_ctx*, long long n, double* y, const double* x);                /* :564-572 */
int hb_vec_component_div(hb_ctx*, long long n, double* y, const double* x);                 /* :574-582 */
int hb_vec_component_div_w_pattern(hb_ctx*, long long n, double* y, const double* x, const double* select); /* :584-592 */
int hb_vec_invert(hb_ctx*, long long n, double* y);                                         /* :852-860 */
int hb_vec_select_pattern(hb_ctx*, long long n, double* y, const double* select);           /* :1063-1071 */
int hb_vec_add_constant(hb_ctx*, long long n, double* y, double c);                         /* :793-797 */
int hb_vec_add_constant_w_pattern(hb_ctx*, long long n, double* y, double c, const double* select); /* :799-804 */
int hb_vec_add_log_barrier_grad(hb_ctx*, long long n, double* y, double alpha, const double* x, const double* select); /* :893-905 */
int hb_vec_add_linear_damping_term(hb_ctx*, long long n, double* y, const double* ixl, const double* ixu,
                                   double alpha, double ct);                                /* :927-944 */
/* reductions: result written to *out_host after a stream sync (and an NCCL all-reduce when a communicator is set,
 * SUM for dot/twonorm^2/onenorm/logbarrier/damping, MAX for infnorm, MIN for min/fraction-to-boundary) */
int hb_vec_dot(hb_ctx*, long long n, const double* x, const double* y, double* out_host);   /* dotProductWith :480-499 */
int hb_vec_twonorm(hb_ctx*, long long n, const double* x, double* out_host);                /* twonorm   :463-478 */
int hb_vec_infnorm(hb_ctx*, long long n, const double* x, double* out_host);                /* infnorm   :501-521 */
int hb_vec_onenorm(hb_ctx*, long long n, const double* x, double* out_host);                /* onenorm   :540-553 */
int hb_vec_min_w_pattern(hb_ctx*, long long n, const double* x, const double* select, double* out_host); /* :821-839 */
int hb_vec_log_barrier(hb_ctx*, long long n, const double* x, const double* select, double* out_host);   /* :863-881 */
int hb_vec_linear_damping_term(hb_ctx*, long long n, const double* x, const double* ixl, const double* ixu,
                               double mu, double kappa_d, double* out_host);                /* :907-925 */
int hb_vec_fraction_to_bdry(hb_ctx*, long long n, const double* x, const double* dx, double tau,
                            const double* select_or_null, double* out_host);                /* :1017-1061 */

/* hiopMatrixDenseRowMajor::timesVec / transTimesVec (src/LinAlg/hiopMatrixDenseRowMajor.cpp:436-528):
 * A is m x n row-major with leading dimension lda (elements). With a communicator the m-vector result of
 * hb_mat_times_vec is all-reduced and beta*y is applied on rank 0 only (:464-467). */
int hb_mat_times_vec(hb_ctx*, int m, long long n, const double* A, long long lda, double beta, double* y, double alpha,
                     const double* x);
int hb_mat_trans_times_vec(hb_ctx*, int m, long long n, const double* A, long long lda, double beta, double* y,
                           double alpha, const double* x);

/* hiopMatrixDenseRowMajor primitives as standalone calls (row-major, leading dimensions in elements; SURVEY 8 a13):
 *   hb_mat_times_mat_trans           C (m x k) = beta C + alpha A (m x n) B (k x n)^T          timesMatTrans_local  :646-674 (local product)
 *   hb_mat_add_sub_diagonal          M[s+i][s+i] += alpha * d[src+i] (d == NULL: += alpha)     addDiagonal / addSubDiagonal :703-764
 *   hb_mat_add_matrix                Y += alpha X                                             addMatrix :766-776
 *   hb_mat_copy_rows_from            dst row i = src row rows_idx[i] (device int indices)      copyRowsFrom :169-197
 *   hb_mat_copy_block                dst block at (dst_i,dst_j) = src block at (src_i,src_j)   copyBlockFromMatrix / copyFromMatrixBlock :200-236
 *   hb_mat_trans_add_to_sym_upper    W(row_start+j, col_start+i) += alpha A(i,j)               transAddToSymDenseMatrixUpperTriangle :779-798
 *   hb_mat_add_upper_to_sym_upper    W diag block += alpha triu(A)                             addUpperTriangleToSymDenseMatrixUpperTriangle :810-829 */
int hb_mat_times_mat_trans(hb_ctx*, int m, int k, long long n, const double* A, long long lda, const double* B, long long ldb, double beta, double* C,
                           long long ldc, double alpha);
int hb_mat_add_sub_diagonal(hb_ctx*, double* M, long long ld, int start_on_dest_diag, int num_elems, double alpha, const double* d_or_null,
                            int start_on_src_vec);
int hb_mat_add_matrix(hb_ctx*, int m, int n, double* Y, long long ldy, double alpha, const double* X, long long ldx);
int hb_mat_copy_rows_from(hb_ctx*, int n_rows, int n_cols, double* dst, long long ldd, const double* src, long long lds, const int* rows_idx_dev);
int hb_mat_copy_block(hb_ctx*, int m, int n, double* dst, long long ldd, int dst_i, int dst_j, const double* src, long long lds, int src_i, int src_j);
int hb_mat_trans_add_to_sym_upper(hb_ctx*, int m, int n, const double* A, long long lda, int row_start, int col_start, double alpha, double* W, long long ldw);
int hb_mat_add_upper_to_sym_upper(hb_ctx*, int n, const double* A, long long lda, int diag_start, double alpha, double* W, long long ldw);

/* ------------------------------------------------------------------------------------------------------------
 * hiopLinSolverSymDense (B1; src/LinAlg/hiopLinSolver.hpp:78-128, LAPACK twin hiopLinSolverSymDenseLapack.hpp:75-192,
 * MAGMA twins hiopLinSolverSymDenseMagma.cpp:120-270, 324-476)
 * ------------------------------------------------------------------------------------------------------------ */
#define HB_FACT_BUNCH_KAUFMAN 0 /* pivoted LDL^T (DSYTRF / magma_dsytrf_gpu semantics), inertia from 1x1/2x2 pivots */
#define HB_FACT_NOPIV 1         /* LDL^T without pivoting (magma_dsytrf_nopiv_gpu, linsol_mode=speculative) */
#define HB_FACT_CHOLESKY 2      /* LL^T for SPD systems (DPOTRF; duals LSQ + condensed QN system) */

int hb_symdense_create(hb_ctx* ctx, int N, hb_symdense** out);
int hb_symdense_destroy(hb_symdense* s);
/* device pointer of the N x N row-major system matrix M_ (sysMatrix(), hiopLinSolver.cpp:99-102); the caller fills
 * its UPPER triangle before each hb_symdense_matrix_changed (hiopKKTLinSysMDS.cpp:196-206). */
double* hb_symdense_matrix(hb_symdense* s);
/* matrixChanged(): factorizes in place. Returns the reference's value: >= 0 number of negative eigenvalues,
 * -1 if a null pivot (|d| < 1e-14, hiopLinSolverSymDenseLapack.hpp:154-166) or a breakdown was met.
 * Values <= -2 are HB_ERR_* codes. */
int hb_symdense_matrix_changed(hb_symdense* s, int mode);
/* inertia of the last factorization (host ints): negative, null, positive */
int hb_symdense_inertia(hb_symdense* s, int* n_neg, int* n_null, int* n_pos);
/* solve(x): in-place solve with nrhs right-hand sides stored one after the other (each N doubles, device).
 * Returns 1 on success, 0 on failure (bool semantics of hiopLinSolver::solve), negative HB_ERR_* on misuse. */
int hb_symdense_solve(hb_symdense* s, double* x, int nrhs);
/* host-buffer convenience used by the C++ adapter when mem_space is host: uploads the upper triangle, factorizes */
int hb_symdense_matrix_changed_host(hb_symdense* s, const double* M_host, int mode);
int hb_symdense_solve_host(hb_symdense* s, double* x_host, int nrhs);
/* diagnostics (tools/prof_diag.py): cycle counters of the phases of the two kernels on the critical path of the large-N factorizations
 * (the 128 x 128 diagonal-block kernel on the leading block of M; the cluster Bunch-Kaufman panel, summed over a factorization) */
int hb_debug_diag128_profile(hb_symdense* s, int ldl, long long* prof_host8);
int hb_debug_bk_profile(hb_ctx* ctx, int on, long long* prof_host8);

/* ------------------------------------------------------------------------------------------------------------
 * hiopKKTLinSysLowRank + hiopHessianLowRank (B2; src/Optimization/hiopKKTLinSys.cpp:1031-1350,
 * src/Optimization/hiopHessianLowRank.cpp:221-630, 974-1059)
 * n_local columns on this rank (all n-vectors and the columns of J, S_t, Y_t are sharded; m-, l-sized data are
 * replicated). m = m_eq + m_ineq constraints, l <= l_max secant pairs.
 * ------------------------------------------------------------------------------------------------------------ */
int hb_lowrank_create(hb_ctx* ctx, long long n_local, int m_eq, int m_ineq, int l_max, hb_lowrank** out);
int hb_lowrank_destroy(hb_lowrank* k);
/* bound patterns ixl, ixu (n_local) and idl, idu (m_ineq): get_ixl()... of hiopNlpFormulation. Borrowed. */
int hb_lowrank_set_patterns(hb_lowrank* k, const double* ixl, const double* ixu, const double* idl, const double* idu);
/* Jacobians Jac_c (m_eq x n_local) and Jac_d (m_ineq x n_local), row-major, leading dimension n_local. Borrowed until
 * the next call. If Jd == Jc + m_eq*n_local the engine uses [Jc;Jd] in place (no copy; the reference copies m x n
 * doubles per solve, hiopKKTLinSys.cpp:1127-1128), otherwise it packs them into an internal m x n_local buffer. */
int hb_lowrank_set_jacobian(hb_lowrank* k, const double* Jc, const double* Jd);
/* Compact-BFGS state as hiopHessianLowRank::update leaves it (hiopHessianLowRank.cpp:262-388): S_t, Y_t are l x n_local
 * row-major device arrays (borrowed); L (l x l row-major, strictly lower) and D (l) are HOST arrays (they are
 * "local" DEFAULT-space objects in the reference too, hiopHessianLowRank.cpp:85-87); sigma = B0 scaling. */
int hb_lowrank_set_secant(hb_lowrank* k, int l, double sigma, const double* St, const double* Yt, const double* L_host,
                          const double* D_host);
/* Secant bookkeeping on the device (hiopHessianLowRank::update, hiopHessianLowRank.cpp:262-388, with growL/growD/updateL/
 * updateD :779-867 and appendRow/shiftRows/replaceRow of hiopMatrixDenseRowMajor.cpp:129-137, 238-284). In this mode the
 * engine OWNS S_t, Y_t, x_prev, grad_f_prev and J_prev; hb_lowrank_set_secant is not called by the host.
 *   hb_lowrank_secant_reset: empty memory, sigma = sigma0; sigma_strategy = HB_SIGMA_* (hiopHessianLowRank.cpp:124-136).
 *   hb_lowrank_secant_update: x, grad_f (n_local), yc, yd = the CURRENT iterate; the current Jacobian is the one registered
 *     with hb_lowrank_set_jacobian. Forms s = x - x_prev and y = grad_f - grad_f_prev + (J - J_prev)^T [yc; yd] in one fused
 *     pass that also refreshes J_prev, applies the reference's two skip rules (||s||_inf < 100 eps; s^T y <= ||s|| ||y||
 *     sqrt(eps)), appends or shifts the pair into S_t / Y_t, updates L, D and sigma (clamped to [1e-8, 1e8]).
 *     jacobian_is_constant != 0 skips the Jacobian terms (linear constraints; no J_prev is allocated).
 *     *status: 0 first iterate stored, 1 pair accepted, 2 skipped (s too small), 3 skipped (s^T y not positive enough).
 *     A stored or accepted pair re-installs the memory like hb_lowrank_set_secant does: call hb_lowrank_update afterwards
 *     (DhInv depends on sigma).
 *   hb_lowrank_secant_state: l, sigma, device pointers of S_t / Y_t (l x n_local row-major), HOST copies of L (l x l) and D. */
#define HB_SIGMA_STY 1
#define HB_SIGMA_STY_INV 2
#define HB_SIGMA_SNRM_YNRM 3
#define HB_SIGMA_STY_SNRM_YNRM 4
#define HB_SIGMA_CONSTANT 5
int hb_lowrank_secant_reset(hb_lowrank* k, double sigma0, int sigma_strategy);
int hb_lowrank_secant_update(hb_lowrank* k, const double* x, const double* grad_f, const double* yc, const double* yd,
                             int jacobian_is_constant, int* status);
int hb_lowrank_secant_state(hb_lowrank* k, int* l, double* sigma, const double** St, const double** Yt, double* L_host, double* D_host);
/* hiopResidual::update (src/Optimization/hiopResidual.cpp:154-368) with the linear damping terms of hiopLogBarProblem
 * (hiopLogBarProblem.hpp:135-145): the 12 residual blocks of the current iterate and its 11 norms in one J^T pass + three fused
 * kernels. it: HOST array of 12 DEVICE pointers {x, d, yc, yd, sxl, sxu, sdl, sdu, zl, zu, vl, vu}; cvals (m_eq), dvals (m_ineq) =
 * constraint bodies, grad_f (n_local), bounds xl, xu (n_local), dl, du (m_ineq), crhs (m_eq); res: 12 DEVICE pointers {rx, rd, ryc,
 * ryd, rxl, rxu, rdl, rdu, rszl, rszu, rsvl, rsvu} as consumed by hb_lowrank_compute_directions; norms_host (11 doubles) =
 * nrmInf {nlp_optim, nlp_feasib, nlp_complem, bar_optim, bar_feasib, bar_complem}, nrmOne {nlp_feasib, bar_feasib, nlp_optim,
 * bar_optim}, nrmInf_cons_violation. Uses the patterns of hb_lowrank_set_patterns and the Jacobian of hb_lowrank_set_jacobian. */
int hb_lowrank_residual_update(hb_lowrank* k, const double* const* it, const double* cvals, const double* dvals, const double* grad_f, double mu,
                               double kappa_d, const double* xl, const double* xu, const double* dl, const double* du, const double* crhs,
                               double* const* res, double* norms_host);
/* Line-search side of one IPM iteration (hiopIterate / hiopLogBarProblem). it / dir / out: HOST arrays of 12 DEVICE pointers in the
 * iterate order {x, d, yc, yd, sxl, sxu, sdl, sdu, zl, zu, vl, vu}; patterns from hb_lowrank_set_patterns.
 *   hb_iterate_fraction_to_bdry: hiopIterate::fractionToTheBdry (hiopIterate.cpp:326-363): largest alpha_primal (slacks) and alpha_dual
 *     (bound duals) with s + alpha ds >= (1 - tau) s; eight reductions of the reference in two fused passes.
 *   hb_iterate_take_step: takeStep_primals (which & 1: x, d) / takeStep_duals (which & 2: yc, yd with alpha_primal; zl, zu, vl, vu
 *     with alpha_dual) (:366-390); out may alias it.
 *   hb_iterate_logbar: hiopLogBarProblem::updateWithNlpInfo (hiopLogBarProblem.hpp:83-120): f_logbar = f - mu sum log(slacks) +
 *     kappa_d mu sum (one-sided slacks), grad_x_logbar = grad_f - mu/sxl + mu/sxu + kappa_d mu (ixl - ixu), grad_d_logbar likewise;
 *     with both gradient pointers NULL it is updateWithNlpInfo_trial_funcOnly (:121-132, function value only).
 *   hb_iterate_adjust_duals_plh: hiopIterate::adjustDuals_primalLogHessian (hiopIterate.cpp:508-521, hiopVectorPar.cpp:1117-1148):
 *     zl, zu, vl, vu are clamped in place to [mu/(kappa_Sigma s), kappa_Sigma mu/s] on their patterns. */
int hb_iterate_fraction_to_bdry(hb_lowrank* k, const double* const* it, const double* const* dir, double tau, double* alpha_primal,
                                double* alpha_dual);
int hb_iterate_take_step(hb_lowrank* k, const double* const* it, const double* const* dir, double alpha_primal, double alpha_dual, int which,
                         double* const* out);
int hb_iterate_adjust_duals_plh(hb_lowrank* k, double* const* it, double mu, double kappa_sigma);
/* hiopIterate::adjust_small_slacks (hiopIterate.cpp:413-505): slacks of `it` that fell below eps*min(1,mu) on their pattern are pushed back
 * (in place) using the bound duals of it_curr and the bounds xl, xu (n_local), dl, du (m_ineq); *num_adjusted = number of adjusted
 * entries on this rank. A block whose smallest slack is not small is left untouched, like in the reference. */
int hb_iterate_adjust_small_slacks(hb_lowrank* k, double* const* it, const double* const* it_curr, double mu, const double* xl, const double* xu,
                                   const double* dl, const double* du, int* num_adjusted);
int hb_iterate_logbar(hb_lowrank* k, const double* const* it, double f, double mu, double kappa_d, const double* grad_f, double* grad_x_logbar,
                      double* grad_d_logbar, double* f_logbar);
/* LSQ multiplier (re)computation hiopDualsLsqUpdateLinsysRedDenseSymPD::do_lsq_update (src/Optimization/hiopDualsUpdater.cpp:
 * 232-332, DPOTRF/DPOTRS :690-735): solves [Jc Jc^T, Jc Jd^T; ., Jd Jd^T + I] [yc; yd] = -[Jc vx; Jd vx + (vl - vu)],
 * vx = grad_f - zl + zu, with the Jacobian registered by hb_lowrank_set_jacobian. J J^T is one pass of the condensation
 * kernel (mode as hb_lowrank_set_condense_mode) + all-reduce; Cholesky on every rank. HB_ERR_NUMERIC if not SPD (the
 * reference then keeps the duals of the line search, hiopDualsUpdater.cpp:263-267). */
int hb_lowrank_lsq_duals(hb_lowrank* k, const double* grad_f, const double* zl, const double* zu, const double* vl, const double* vu,
                         double* yc, double* yd);
/* update(): Dx = zl/sxl|ixl + zu/sxu|ixu, DhInv = 1/(sigma+Dx), Dd = vl/sdl|idl + vu/sdu|idu, Dd_inv = 1/Dd in ONE fused
 * pass (hiopKKTLinSys.cpp:1057-1094 + hiopHessianLowRank.cpp:221-233; 7 n-passes in the reference). Borrows the
 * iterate pointers until the next update (they are read again by hb_lowrank_compute_directions). */
int hb_lowrank_update(hb_lowrank* k, const double* zl, const double* sxl, const double* zu, const double* sxu,
                      const double* vl, const double* sdl, const double* vu, const double* sdu);
/* Forms V (2l x 2l), factorizes it (Bunch-Kaufman), forms N = J (B_k+D_x)^{-1} J^T + blkdiag(0, Dd_inv) with ONE pass
 * over J (fused W, S1, Y1, V-blocks; FP64 tensor-core SYRK), all-reduces it across ranks and Cholesky-factorizes it
 * with equilibration (symMatTimesInverseTimesMatTrans hiopHessianLowRank.cpp:549-630, updateInternalBFGSRepresentation
 * :400-485, DPOSVX('E') hiopKKTLinSys.cpp:1228). The factor is cached until the next update/set_* call.
 * Returns HB_ERR_NUMERIC if N is not numerically SPD. */
int hb_lowrank_condense(hb_lowrank* k);
/* How the GEMM-shaped part of the condensation is computed:
 *   HB_CONDENSE_FP64_DMMA (0): exact FP64 on the DMMA pipe (mma.sync.m8n8k4.f64);
 *   6, 7, 8: INT8-slice (Ozaki) emulation on the tcgen05 tensor cores with that many 7-bit slices -- exact integer
 *   products/accumulation in TMEM, truncation of the operands 2^-41 / 2^-48 / 2^-55 relative to each row's largest entry. */
#define HB_CONDENSE_AUTO (-1)      /* default: 8 slices on tcgen05 when the GLOBAL n (summed over the ranks) >= 32768 and m+2l >= 64, FP64 DMMA otherwise */
#define HB_CONDENSE_FP64_DMMA 0
int hb_lowrank_set_condense_mode(hb_lowrank* k, int mode);
/* Memory of the int8-slice modes. The slices of all n_local columns take S * Mpad * Kpad bytes (Mpad = m+2l rounded up to 128, Kpad =
 * n_local rounded up to 128): as much as the Jacobian in FP64 at S = 8. The context allocates them once when they fit its budget; otherwise
 * it slices and multiplies the columns in chunks of a whole number of int32-safe recombination chunks (65 408 columns at S = 8, 74 880 at
 * S = 7, 87 296 at S = 6) through one buffer of S * Mpad * chunk bytes. The digits are the same either way (row exponents come from all
 * columns); only the grouping of the FP64 partial sums differs, at rounding level.
 * The budget: hb_ctx_set_oz_workspace_limit(ctx, bytes), or the environment variable HB_OZ_WORKSPACE_MB read when the context is created;
 * 0 (the default) = AUTO: the free device memory minus 1 GiB, plus the slice buffer already held. Setting a limit below the buffer held
 * releases it. When not even one recombination chunk (or all columns, when fewer) fits, HB_CONDENSE_AUTO redoes the condensation with the
 * FP64 kernel (counted by hb_lowrank_fallback_count); an explicit 6/7/8 mode fails with HB_ERR_ALLOC.
 * hb_lowrank_last_condense_chunks: column chunks of the last condensation, 1 = unchunked, 0 = the FP64 kernel ran. */
int hb_ctx_set_oz_workspace_limit(hb_ctx* ctx, size_t bytes);
int hb_lowrank_last_condense_chunks(hb_lowrank* k);
/* hb_lowrank_condense is synchronous: it returns HB_ERR_NUMERIC when V is singular or N is not numerically SPD. In AUTO mode an
 * int8-slice condensation whose Cholesky breaks down, or whose slices do not fit (above), is first redone with the exact FP64 kernel
 * (hb_lowrank_fallback_count counts these). hb_lowrank_condense_async only enqueues the work (no host synchronisation; this is also what an implicit condensation
 * inside hb_lowrank_solve_compressed does); a breakdown is then reported by hb_lowrank_check / hb_lowrank_last_solve_stats, the next
 * calls that synchronise. */
int hb_lowrank_condense_async(hb_lowrank* k);
int hb_lowrank_check(hb_lowrank* k);
int hb_lowrank_fallback_count(hb_lowrank* k);
/* the mode the last hb_lowrank_condense actually used (0, 6, 7 or 8) */
int hb_lowrank_get_condense_mode(hb_lowrank* k);
/* solveCompressed(rx,ryc,ryd -> dx,dyc,dyd) (hiopKKTLinSys.cpp:1110-1190) incl. the residual-driven refinement of
 * solveWithRefin (:1192-1350: ||rhs - N x||_inf < 1e-8, <= 3 corrections). Condenses first if the cache is stale.
 * Like the reference, rx is used as scratch and overwritten (:1178). */
int hb_lowrank_solve_compressed(hb_lowrank* k, double* rx, const double* ryc, const double* ryd, double* dx, double* dyc,
                                double* dyd);
/* computeDirections (hiopKKTLinSysCompressedXYcYd::computeDirections hiopKKTLinSys.cpp:585-691 +
 * compute_directions_for_full_space :218-309): the 12 residual blocks -> the 12 direction blocks.
 * res = {rx, rd, ryc, ryd, rxl, rxu, rdl, rdu, rszl, rszu, rsvl, rsvu}; dir = {x, d, yc, yd, sxl, sxu, sdl, sdu, zl, zu, vl, vu}
 * (HOST arrays of 12 DEVICE pointers). Residuals are not modified. */
int hb_lowrank_compute_directions(hb_lowrank* k, const double* const* res, double* const* dir);
/* compute_directions_w_IR (hiopKKTLinSys::compute_directions_w_IR hiopKKTLinSys.cpp:909-960): BiCGStab
 * (hiopBiCGStabSolver::solve, src/LinAlg/hiopKrylovSolver.cpp:399-700; same recurrence, breakdown / stagnation / "more
 * steps" rules and minimal-residual fallback) on the unreduced 12-block KKT system with hb_lowrank_compute_directions as
 * the preconditioner and x0 = 0. res / dir as in hb_lowrank_compute_directions. tol is the RELATIVE tolerance the
 * reference computes as min(mu*ir_outer_tol_factor, ir_outer_tol_min) (:942); maxit = ir_outer_maxit (<= 0: plain
 * computeDirections, :914-917). info (HOST, 4 doubles, may be NULL) = {flag (0 converged, 3 stagnation, 4 breakdown,
 * 1 iteration limit), iterations (half steps count 0.5), abs residual, rel residual}. Like the reference the step is
 * accepted whatever the flag (:950-953), so the return value reports only engine errors. */
int hb_lowrank_compute_directions_w_ir(hb_lowrank* k, const double* const* res, double* const* dir, double tol, int maxit, double* info);
/* y = K x with the full (unsymmetric) 12 x 12 block KKT operator hiopMatVecKKTFullOpr::times_vec
 * (hiopKKTLinSys.cpp:1619-1733); x, y: HOST arrays of 12 DEVICE pointers in the order of dir / res above. */
int hb_lowrank_kkt_full_times_vec(hb_lowrank* k, const double* const* x, double* const* y);
/* hiopKKTLinSysCompressed::test_direction (hiopKKTLinSys.cpp:455-509) for the low-rank Hessian: dWd = dx^T (B_k + D_x + delta_wx) dx +
 * dd^T (D_d + delta_wd) dd against neg_curv_test_fact (||dx||^2 + ||dd||^2). delta_* may be NULL (the quasi-Newton driver runs with
 * hiopPDPerturbationNull). out_host2 = {dWd, ||dx||^2 + ||dd||^2}. Returns 1 (accept), 0 (negative curvature), < 0 on error. */
int hb_lowrank_test_direction(hb_lowrank* k, const double* dx, const double* dd, const double* delta_wx, const double* delta_wd, double neg_curv_test_fact,
                              double* out_host2);
/* x = (B_k + D_x)^{-1} rhs  (hiopHessianLowRank::solve :495-540) */
int hb_lowrank_hess_solve(hb_lowrank* k, const double* rhs, double* x);
/* y = beta*y + alpha*(B_k [+ D_x]) x in the compact form (same operator as the recursive timesVecCmn :974-1059) */
int hb_lowrank_hess_times_vec(hb_lowrank* k, double beta, double* y, double alpha, const double* x, int add_log_term);
/* read-backs (device pointers owned by the engine; valid until destroy): Dx, DhInv (n_local), Dd_inv (m_ineq),
 * N (m x m row-major, full symmetric storage, UNfactorized copy) */
const double* hb_lowrank_Dx(hb_lowrank* k);
const double* hb_lowrank_DhInv(hb_lowrank* k);
const double* hb_lowrank_Dd_inv(hb_lowrank* k);
const double* hb_lowrank_N(hb_lowrank* k);
/* statistics of the last solve: refinement steps taken, last residual inf-norm (host) */
int hb_lowrank_last_solve_stats(hb_lowrank* k, int* n_refine, double* resid_inf);
/* One whole KKT system from HOST buffers (the e2e path of bench.py and of the C++ adapter when HiOp keeps its data in
 * host memory): H2D of the iterate blocks, (optionally) J and rhs, update + condense + solve, D2H of dx,dyc,dyd.
 * J_host may be NULL to reuse the device-resident Jacobian from the previous call. */
int hb_lowrank_kkt_system_host(hb_lowrank* k, const double* Jc_host, const double* Jd_host, const double* zl,
                               const double* sxl, const double* zu, const double* sxu, const double* vl, const double* sdl,
                               const double* vu, const double* sdu, const double* rx, const double* ryc, const double* ryd,
                               double* dx, double* dyc, double* dyd);

/* ------------------------------------------------------------------------------------------------------------
 * hiopKKTLinSysCompressedMDSXYcYd (src/Optimization/hiopKKTLinSysMDS.cpp:59-484): mixed dense-sparse Newton KKT.
 * x = (x_s, x_d) with nxs "sparse" and nxd "dense" variables; the Hessian is diag(H_s) (+) H_d, the Jacobians are
 * [J_s | J_d] with J_s sparse triplets (row-sorted) and J_d dense row-major. The condensed system has size
 * N = nxd + neq + nineq and is handed to an hb_symdense solver. Stays on one GPU.
 * ------------------------------------------------------------------------------------------------------------ */
int hb_mds_create(hb_ctx* ctx, int nxs, int nxd, int neq, int nineq, hb_mds** out);
int hb_mds_destroy(hb_mds* h);
/* sparsity of Jac_c_sp (neq x nxs) and Jac_d_sp (nineq x nxs): HOST triplet index arrays sorted by (row, col)
 * (hiopMatrixSparseTriplet's ordering assumption, src/LinAlg/hiopMatrixSparseTriplet.cpp:528-560). Static per problem. */
int hb_mds_set_sparsity(hb_mds* h, int nnz_c, const int* iRow_c_host, const int* jCol_c_host, int nnz_d, const int* iRow_d_host,
                        const int* jCol_d_host);
/* update(): Dx = zl/sxl|ixl + zu/sxu|ixu over all nxs+nxd variables (hiopKKTLinSysMDS.cpp:155-157) */
int hb_mds_update(hb_mds* h, const double* zl, const double* sxl, const double* zu, const double* sxu, const double* ixl, const double* ixu);
/* build_kkt_matrix() (:172-305): fills the UPPER triangle of Msys (N x N row-major, e.g. hb_symdense_matrix(s)) with
 *   [ Hd + Dxd + dwx     Jcd^T                         Jdd^T                                  ]
 *   [                   -Jcs Hxs^{-1} Jcs^T - dcc      -Jcs Hxs^{-1} Jds^T                    ]
 *   [                                                  -Jds Hxs^{-1} Jds^T - Dd_inv - dcd     ]
 * Hxs = Dxs + dwx + diag(H_s), Dd_inv = 1/(dwd + vl/sdl|idl + vu/sdu|idu). Hd: nxd x nxd (upper triangle read),
 * Hs_diag: nxs, Jcd: neq x nxd, Jdd: nineq x nxd, J*s_vals: nnz values in triplet order, delta_wx: nxs+nxd,
 * delta_wd/delta_cd: nineq, delta_cc: neq (the regularisations arrive as vectors, hiopPDPerturbation.hpp:113-134). */
int hb_mds_build_kkt_matrix(hb_mds* h, const double* Hd, const double* Hs_diag, const double* Jcd, const double* Jdd,
                            const double* Jcs_vals, const double* Jds_vals, const double* vl, const double* sdl, const double* vu,
                            const double* sdu, const double* idl, const double* idu, const double* delta_wx, const double* delta_wd,
                            const double* delta_cc, const double* delta_cd, double* Msys);
/* Haynsworth part of factorizeWithCurvCheck (:78-110): #entries of Hxs < -1e-14 and #entries with |.| < 1e-14 (host ints) */
int hb_mds_hxs_inertia(hb_mds* h, int* n_neg, int* n_zero);
/* solveCompressed() (:307-403) around s (already factorized with hb_symdense_matrix_changed). rx has nxs+nxd entries. */
int hb_mds_solve_compressed(hb_mds* h, hb_symdense* s, const double* rx, const double* ryc, const double* ryd, double* dx, double* dyc,
                            double* dyd);
/* ---- dense-Newton KKT classes hiopKKTLinSysDenseXYcYd (form 0) / hiopKKTLinSysDenseXDYcYd (form 1) ----
 * build_kkt_matrix (src/Optimization/hiopKKTLinSysDense.hpp:85-172, 249-330): fills Msys (N x N row-major, upper triangle;
 * N = nx+neq+nineq, resp. nx+2*nineq+neq) with [H+Dx+dwx, Jc^T, Jd^T; 0; -Dd^{-1}] resp. [H+Dx+dwx, 0, Jc^T, Jd^T; Dd+dwd, 0, -I;
 * ...]. Dx = zl/sxl|ixl + zu/sxu|ixu and Dd (form 1) or Dd_inv = 1/(dwd + vl/sdl|idl + vu/sdu|idu) (form 0) are computed
 * like update() does and returned in the caller's Dx (nx) / Dd (nineq) buffers. As in the reference, delta_cd is subtracted
 * from the nineq diagonal entries starting at the FIRST dual row (:157, :312) and delta_cc is not used.
 * solveCompressed (:174-207, :332-370): stack the blocks, hb_symdense_solve, split. work: N doubles. rd/dd: form 1 only. */
int hb_densekkt_build(hb_ctx* ctx, int form, int nx, int neq, int nineq, const double* H, const double* Jc, const double* Jd,
                      const double* zl, const double* sxl, const double* zu, const double* sxu, const double* ixl, const double* ixu,
                      const double* vl, const double* sdl, const double* vu, const double* sdu, const double* idl, const double* idu,
                      const double* delta_wx, const double* delta_wd, const double* delta_cc, const double* delta_cd, double* Dx,
                      double* Dd, double* Msys);
int hb_densekkt_solve_compressed(hb_ctx* ctx, hb_symdense* s, int form, int nx, int neq, int nineq, const double* rx, const double* rd,
                                 const double* ryc, const double* ryd, double* dx, double* dd, double* dyc, double* dyd, double* work);
/* ---- write_kkt interchange files (.iajaaa): hiopCSR_IO::writeMatToFile / writeRhsToFile / writeSolToFile
 * (src/Utils/hiopCSR_IO.hpp:44-155), format in src/LinAlg/csr_iajaaa.md. Byte-compatible with the reference writer. M: N x N
 * row-major, upper triangle (what build_kkt_matrix leaves in sysMatrix() BEFORE matrixChanged()); vectors are appended one per
 * line (rhs, then solution, repeatable). *_host take host arrays and need no GPU; the others download from the device. */
int hb_iajaaa_write_matrix_host(const char* filename, int N, const double* M_host, int nx, int meq, int mineq);
int hb_iajaaa_append_vector_host(const char* filename, int N, const double* v_host);
int hb_iajaaa_write_matrix(hb_ctx* ctx, const char* filename, int N, const double* M_dev, int nx, int meq, int mineq);
int hb_iajaaa_append_vector(hb_ctx* ctx, const char* filename, int N, const double* v_dev);
const double* hb_mds_Dx(hb_mds* h);
const double* hb_mds_Hxs(hb_mds* h);
const double* hb_mds_Dd_inv(hb_mds* h);

#ifdef __cplusplus
}
#endif
#endif /* HIOPB200_H */
