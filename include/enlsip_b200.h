/* enlsip_b200.h -- C ABI of the B200-native ENLSIP Gauss-Newton engine (batched regime).
 *
 * Drop-in boundary for the reference call site
 *     solve!(model) -> enlsip(x0, r, c, n, m, q, l; scaling, MAX_ITER, TIME_LIMIT, eps_rel, eps_x, eps_c, eps_rank)
 *                   -> (exit_code, x_opt, f_opt, ExecutionInfo)
 * (reference src/solver.jl:80-87, src/enlsip_functions.jl:2638-2655, 2879).  The Julia host layer
 * (julia/EnlsipB200.jl) binds these symbols with `ccall`; tests bind them with ctypes.
 *
 * The reference's plugin surface -- four Julia closures wrapped by ResidualsFunction /
 * ConstraintsFunction (src/cnls_model.jl:11-62) -- cannot cross a C ABI to a GPU.  It is replaced
 * by a `family` id (a device functor compiled into the library) plus device/host data arrays.
 * Constraint order and 1-based constraint ids are the reference's:
 *     [equalities; inequalities; x - x_low (finite entries, index order); x_upp - x (finite entries)]
 * (src/cnls_model.jl:402-403, 416).
 *
 * All functions return 0 on success or a negative ENLSIPB200_E* code; algorithmic outcomes are
 * values in the per-problem `exit_code[]` (raw EF code, src/enlsip_functions.jl:2371-2396) and
 * `status[]` (after convert_exit_code, src/cnls_model.jl:166-178).  Nothing throws.  There is no
 * CPU fallback: every compute entry point fails with ENLSIPB200_ENOGPU when no CUDA device exists.
 */
#ifndef ENLSIP_B200_H
#define ENLSIP_B200_H
/* Every entry point is exported explicitly; the libraries are built with -fvisibility=hidden so that nothing else (template
 * instantiations, inline functions with static state) is shared between the stock library and the libraries that
 * enlsipb200_compile_family / enlsipb200_large_compile_family build -- several of them live in one process. */
#if defined(__GNUC__)
#define ENLSIPB200_API __attribute__((visibility("default")))
#else
#define ENLSIPB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define ENLSIPB200_FAMILY_HS65 0         /* test/problems/HS65.jl:7-17 ; n=3 m=3, 1 inequality       */
#define ENLSIPB200_FAMILY_GAUSS_PEAKS 1  /* BASELINE.json config 3 ; n=6 m=128, 1 equality            */
#define ENLSIPB200_FAMILY_OSBORNE2 2     /* test/problems/osborne2.jl ; n=11 m=65, bounds only          */
#define ENLSIPB200_FAMILY_CHAINED_ROSENBROCK10 3 /* test/problems/chained_rosenbrock.jl with n=10 (m=18, q=8) */
#define ENLSIPB200_FAMILY_CHAINED_WOOD20 4       /* test/problems/chained_wood.jl, n=20 (m=54, q=13)          */

#define ENLSIPB200_JAC_ANALYTIC 0
#define ENLSIPB200_JAC_FORWARD_DIFF 1    /* src/cnls_model.jl:65-82                                    */

#define ENLSIPB200_EINVAL -1
#define ENLSIPB200_ENOGPU -2
#define ENLSIPB200_ECUDA -3
#define ENLSIPB200_ENOMEM -4

/* extra per-problem exit codes (besides the reference's, EF:2371-2396) */
#define ENLSIPB200_EXIT_WOULD_THROW -99  /* the reference raises a Julia exception at this point      */
#define ENLSIPB200_EXIT_WOULD_HANG -98   /* the reference loops forever at this point (EF:621-647)    */
#define ENLSIPB200_EXIT_CAPACITY -97     /* batched regime only: initial working set larger than       */
                                         /* min(lmax, n); x = x0, f = ||r(x0)||^2, iterations 0, nact / */
                                         /* active = the whole initial working set, counters = {2, 2}   */
                                         /* (the one evaluation of r, c, J and A at x0: unlike -11 with */
                                         /* time_limit < 0, which reports 0).  The large regime has no  */
                                         /* such limit (its buffers grow with the working set).         */

#define ENLSIPB200_TRACE_HDR 16          /* doubles per trace row before the n iterate entries         */

/* keyword arguments of solve! (src/solver.jl:62-63).  A NaN tolerance means "reference default":
 * abs_tol = eps, rel_tol = sqrt(abs_tol), c_tol = x_tol = rel_tol.  As in the reference, abs_tol
 * is used only to derive rel_tol (it is never forwarded to enlsip, SURVEY.md T4). */
typedef struct enlsipb200_options {
    int max_iter;        /* 100   */
    int scaling;         /* 0     */
    int jac_mode;        /* ENLSIPB200_JAC_*  (the reference's default is AD = analytic to rounding) */
    int reserved;
    double time_limit;   /* 1e3 seconds */
    double abs_tol, rel_tol, c_tol, x_tol;
} enlsipb200_options;

typedef struct enlsipb200_handle_s* enlsipb200_handle;

ENLSIPB200_API int enlsipb200_version(void);
ENLSIPB200_API const char* enlsipb200_last_error(void);
ENLSIPB200_API void enlsipb200_default_options(enlsipb200_options* opt);

/* problem family + bounds (replaces CnlsModel(...) + instantiate_constraints_*; cnls_model.jl:345-496).
 * x_low / x_upp: host arrays of length n, +-Inf = no bound.  device < 0 = current device. */
ENLSIPB200_API int enlsipb200_create(int family, const double* x_low, const double* x_upp, int device, enlsipb200_handle* out);
ENLSIPB200_API int enlsipb200_destroy(enlsipb200_handle h);
ENLSIPB200_API int enlsipb200_dims(enlsipb200_handle h, int* n, int* m, int* nb_eq, int* nb_constraints, int* lmax);

/* family data arrays (GAUSS_PEAKS: slot 0 = y [B,128], slot 1 = S [B]; OSBORNE2: slot 0 = t [65], slot 1 = y [65],
 * shared by the whole batch).  `on_device` != 0: ptr is a device pointer that must stay valid for the solve.
 * Otherwise ptr is a HOST buffer that must stay valid until the next enlsipb200_solve_batch returns: the upload
 * happens inside that call -- with host-buffer solves chunk by chunk, overlapped with the solves of the previous
 * chunk (pinned host memory makes the copies asynchronous). */
ENLSIPB200_API int enlsipb200_set_data(enlsipb200_handle h, int slot, const double* ptr, long long count, int on_device, void* stream);

/* solve B independent problems (replaces B calls of solve!).  All array arguments are host or
 * device pointers according to `on_device`; optional outputs may be NULL.
 *   x0 [B,n] starting points;  x [B,n] x_opt;  f [B] sum of squared residuals (obj_value);
 *   exit_code/status/iters/nact [B];  active [B,lmax] 1-based ids of the final working set;
 *   counters [B,2] nb_function_evaluations, nb_jacobian_evaluations (reference counting formula);
 *   trace [B,trace_cap,TRACE_HDR+n] per-iteration records (tests only).
 * Blocking unless on_device != 0 and a stream is given (then enqueued on that stream). */
ENLSIPB200_API int enlsipb200_solve_batch(enlsipb200_handle h, long long B, const double* x0, const enlsipb200_options* opt,
                           double* x, double* f, int* exit_code, int* status, int* iters, int* nact, int* active,
                           int* counters, double* trace, int trace_cap, int on_device, void* stream);

/* measurement hooks: device time of the last solve kernel (CUDA events on its stream), launch
 * geometry, number of kernels launched by this handle so far */
ENLSIPB200_API int enlsipb200_last_kernel_ms(enlsipb200_handle h, float* ms);
ENLSIPB200_API int enlsipb200_kernel_info(enlsipb200_handle h, int* regs_per_thread, int* smem_bytes_per_cta, int* threads_per_cta,
                           int* ctas_per_sm, int* grid, int* lanes_per_problem);
/* The evaluation layer as an operator of its own: new_point! (src/enlsip_functions.jl:34-52) through the wrappers
 * res_eval! / jacres_eval! / cons_eval! / jaccons_eval! (src/cnls_model.jl:40-62), with jac_forward_diff
 * (src/cnls_model.jl:65-82) when opt->jac_mode = ENLSIPB200_JAC_FORWARD_DIFF.  DEVICE buffers only:
 *   x [B, n] in;  r [B, m];  J [B, n, m] (per problem the m x n Jacobian, column major as in the reference);
 *   c [B, lmax];  A [B, lmax, n] (row i = gradient of constraint i, bound rows +-e_j included).  Any output may be NULL.
 * enlsipb200_last_kernel_ms reports the kernel time. */
ENLSIPB200_API int enlsipb200_eval_batch(enlsipb200_handle h, long long B, const double* x, const enlsipb200_options* opt, double* r,
                          double* J, double* c, double* A, int on_device, void* stream);
/* One Gauss-Newton step per problem from MATERIALISED inputs -- the batched step kernel of the coalesced-load design:
 * update_working_set (src/enlsip_functions.jl:686-795: qr(A_active', ColumnNorm()), first-order multipliers, J*Q1,
 * qr(J2, ColumnNorm()), the triangular solves of sub_search_direction :116-153, second-order multipliers :514-537 and a
 * possible deletion) applied to r [B, m], J [B, n, m], c [B, lmax], A [B, lmax, n] in the layout enlsipb200_eval_batch
 * writes, from the working set of init_working_set (:826-859).  Outputs: p [B, n] (Gauss-Newton direction), lam
 * [B, min(lmax, n)] (multipliers in working-set order, 0 padded; may be NULL), active [B, lmax] (may be NULL),
 * info [B, 5] = {t, rankA, rankJ2, index_del, error code (0, -99, -97)} (may be NULL).  A problem with a nonzero error
 * code gets p = 0 and lam = 0; with -97, t and active are the whole initial working set.  DEVICE buffers only. */
ENLSIPB200_API int enlsipb200_step_batch(enlsipb200_handle h, long long B, const double* x, const double* r, const double* J,
                                         const double* c, const double* A, const enlsipb200_options* opt, double* p, double* lam,
                                         int* active, int* info, int on_device, void* stream);
ENLSIPB200_API long long enlsipb200_launch_count(enlsipb200_handle h);

/* Run-time compiled problem family: the replacement of the reference's plugin surface -- `residuals`,
 * `eq_constraints`, `ineq_constraints` and their optional `jacobian_*` closures handed to CnlsModel(...)
 * (src/cnls_model.jl:345-359, wrapped at :11-62).  `source` is CUDA C++ defining, in namespace enl_user,
 *     __device__ double residual(int i, const double* x, const double* d0, const double* d1, const double* d2);
 *     __device__ void   constraints(const double* x, const double* d0, const double* d1, const double* d2, double* c);
 *         c[0..nb_eq) equalities then c[nb_eq..nb_eq+nb_ineq) inequalities (>= 0)   (order of cnls_model.jl:402-403)
 * and, if has_jacobians != 0,
 *     __device__ void jac_residual(int i, const double* x, const double*, const double*, const double*, double* grad);                  -- grad[n]
 *     __device__ void jac_constraints(const double* x, const double*, const double*, const double*, double* A);   -- A[(nb_eq+nb_ineq) x n], row major
 * d0 / d1: this problem's rows of data slots 0 / 1 (stride0 / stride1 doubles per problem); d2: slot 2, shared by the batch.
 * The helpers of csrc/enl_base.h (det_exp, det_tanh, add_rn, ...) are visible.  Without Jacobians the solve must use
 * ENLSIPB200_JAC_FORWARD_DIFF (cnls_model.jl:65-82).  Bounds are given to enlsipb200_create as for any family.
 * nvcc (PATH or $ENLSIP_NVCC) compiles the solver for this family into `out_lib_path`; the host then loads THAT library
 * and uses this same API with family = ENLSIPB200_FAMILY_USER.  `work_dir`: writable directory for the generated
 * prelude and the build log.  Limits: n <= 32, m <= 4096, nb_eq + nb_ineq <= 32. */
#define ENLSIPB200_FAMILY_USER 64
ENLSIPB200_API int enlsipb200_compile_family(const char* source, int n, int m, int nb_eq, int nb_ineq, int stride0, int stride1,
                              int has_jacobians, const char* out_lib_path, const char* work_dir);

/* The same plugin surface for the large regime (one problem, n + m >= 1000).  `source` defines, in namespace enl_user,
 *     template <class X> __device__ double residual(long long i, int n, const X& x, const double* d0, const double* d1);
 *     template <class X> __device__ double constraint(int k, int n, const X& x, const double* d0, const double* d1);
 *         k < nb_eq: equalities, then the inequalities (>= 0); X is a point accessor, x[j]
 * and, if has_jacobians != 0,
 *     __device__ double jac_residual(long long i, int j, int n, const double* x, const double* d0, const double* d1);
 *     __device__ double jac_constraint(int k, int j, int n, const double* x, const double* d0, const double* d1);
 * (entry (i, j) of the dense Jacobian).  d0 / d1: the two data slots of enlsipb200_large_set_data (any length).  The
 * helpers of csrc/enl_base.h are visible in namespace enl (enl::det_tanh, ...); ENL_LUSER_M holds m.
 * The resulting library exports the enlsipb200_large_* API; create the handle with family = ENLSIPB200_FAMILY_USER,
 * m_local = m_global = m, any n >= 3 (nb / ineq / rho ignored), bounds through x_low / x_upp.  Without Jacobians the
 * solve differentiates by forward differences (cnls_model.jl:65-82). */
ENLSIPB200_API int enlsipb200_large_compile_family(const char* source, long long m, int nb_eq, int nb_ineq, int has_jacobians,
                                    const char* out_lib_path, const char* work_dir);

/* deterministic exp used by the synthetic families, exposed for bit-parity tests vs oracle/detmath.c */
ENLSIPB200_API int enlsipb200_det_exp(const double* x, double* y, long long n, int on_device);

/* ===========================================================================================
 * Large-Jacobian regime (BASELINE.json configs 4/5): ONE problem whose m x n residual Jacobian is
 * too large for a CTA.  Replaces the same reference call site (solve! -> enlsip, src/solver.jl:80-87);
 * per iterate the engine factors [J | r] with a tall-skinny Householder QR on the GPU
 * (replacing `qr(J2, ColumnNorm())` and `F.Q' * v`, src/enlsip_functions.jl:135-151, 219-223) and
 * runs the pivoted small-matrix stage on the (n+1) x (n+1) triangular factor.
 *
 * Rows may be sharded over several GPUs / processes (one handle per GPU): every rank passes its own
 * m_local rows of W and y and the global m; the ranks are joined by enlsipb200_large_comm_init
 * (NCCL: all-gather of the per-GPU R factors, all-reduce of the linesearch sums).  Every rank then
 * calls enlsipb200_large_solve with the same x0 / options and receives the same results.
 * =========================================================================================== */
#define ENLSIPB200_FAMILY_SINGLE_INDEX 16 /* r_i = det_tanh(w_i.x) - y_i ; block constraints on groups of 4
                                             parameters: equalities sum x_j^2 - rho_k (ineq = 0) or
                                             inequalities rho_k - sum x_j^2 >= 0 (ineq = 1); optional bounds */

#define ENLSIPB200_FAMILY_LARGE_CHAINED_ROSENBROCK 17 /* test/problems/chained_rosenbrock.jl:8-53 at ANY n (the reference
                                             runs n = 1000: m = 2(n-1) = 1998 residuals, q = n-2 = 998 nonlinear
                                             equalities); a general "row family": no restriction on n; analytic or
                                             forward-difference Jacobians (opt->jac_mode); nb / ineq / rho are ignored.
                                             m_local = m_global = 2(n-1), unless ENLSIPB200_LARGE_FACTOR_TSQR is set:
                                             then the rows may be sharded (m_local <= m_global)                       */

/* OR-ed into `family` of enlsipb200_large_create.  Row families (built-in or ENLSIPB200_FAMILY_USER) then build [J | r]
 * row major, with n padded to a multiple of 32 by zero columns, and compress it with the tall-skinny QR of the
 * single-index family instead of the plain Householder QR of a column-major [J | r].  The rows may then be sharded over
 * GPUs: each rank passes its own m_local <= m_global = m(n) rows, enlsipb200_large_comm_init places the shards in rank
 * order (row0 = the rows of the lower ranks) and refuses, on every rank, a total other than m_global.  Data slots stay
 * whole on every rank and the family is called with global row indices.  The single-index family accepts the flag and
 * ignores it. */
#define ENLSIPB200_LARGE_FACTOR_TSQR 0x100

typedef struct enlsipb200_large_s* enlsipb200_large;

ENLSIPB200_API const char* enlsipb200_large_last_error(void);

/* n: parameters (multiple of 32); m_local: residual rows held by this handle; m_global: all rows;
 * nb: number of 4-parameter blocks with a constraint; rho [nb]; x_low / x_upp [n] or NULL (+-Inf = none). */
ENLSIPB200_API int enlsipb200_large_create(int family, int n, long long m_local, long long m_global, int nb, int ineq,
                            const double* rho, const double* x_low, const double* x_upp, int device,
                            enlsipb200_large* out);
ENLSIPB200_API int enlsipb200_large_destroy(enlsipb200_large h);
/* slot 0 = W [m_local, n] row major, slot 1 = y [m_local].  on_device != 0: device pointer that must stay
 * valid (and resident on the handle's device) for the solves; otherwise copied host -> device. */
ENLSIPB200_API int enlsipb200_large_set_data(enlsipb200_large h, int slot, const double* ptr, long long count, int on_device);
/* multi-GPU: rank 0 creates a 128-byte NCCL unique id, the host layer distributes it, every rank joins.  A row family
 * created with ENLSIPB200_LARGE_FACTOR_TSQR and m_local < m_global must join before its first solve or factor. */
ENLSIPB200_API int enlsipb200_large_comm_id(void* id128);
ENLSIPB200_API int enlsipb200_large_comm_init(enlsipb200_large h, const void* id128, int rank, int nranks);
/* blocking solve; outputs as in enlsipb200_solve_batch for B = 1 (active [l], trace [trace_cap, TRACE_HDR + n]) */
ENLSIPB200_API int enlsipb200_large_solve(enlsipb200_large h, const double* x0, const enlsipb200_options* opt, double* x, double* f,
                           int* exit_code, int* status, int* iters, int* nact, int* active, double* trace,
                           int trace_cap);
/* measurement / test hook: evaluate [J | r] at x and factor it; R [(n+1) x (n+1)] row major (may be NULL);
 * device times of the two stages (CUDA events on the handle's stream) */
ENLSIPB200_API int enlsipb200_large_factor(enlsipb200_large h, const double* x, double* R, float* build_ms, float* tsqr_ms);
/* cumulative counters: {points evaluated (new_point!), build ms, tsqr ms, linesearch ms, solve wall ms, linesearch
 * evaluations (host clock around launch..result), kernels launched, padded local rows, device QRCPs, device M*Q products,
 * ms inside the small-stage calls (host clock: kernels + the waits for their results), factorisations of [J | r] (one per
 * point from which the iteration continued), growths of the working-set buffers (a working set of more than
 * min(l, n) + 1 rows)}; `count` may stop short of the last entries */
ENLSIPB200_API int enlsipb200_large_stats(enlsipb200_large h, double* out, int count);

/* Known-answer hooks of the small stage's dense kernels (csrc/enl_small.cuh), host buffers, column major:
 *   enlsipb200_dense_qrcp : `qr(M, ColumnNorm())` of src/enlsip_functions.jl:223 / :700 / :769 = LAPACK dgeqp3
 *       f [rows x cols] in/out (dgeqp3 layout: R above, reflectors below the diagonal), tau [min(rows, cols)],
 *       jpvt [cols] 0-based;
 *   enlsipb200_dense_mulq : `J * F_A.Q` of src/enlsip_functions.jl:219: M [mr x nq] <- M * H(0) ... H(k-1), the
 *       reflectors in f [nq x k] / tau [k] (dgeqp3 layout). */
ENLSIPB200_API int enlsipb200_dense_qrcp(int rows, int cols, double* f, double* tau, int* jpvt, int device);
/*   enlsipb200_dense_qr : the plain Householder QR (LAPACK dgeqrf, no pivoting) that compresses [J | r] of the general
 *       large-regime families; f / tau as enlsipb200_dense_qrcp. */
ENLSIPB200_API int enlsipb200_dense_qr(int rows, int cols, double* f, double* tau, int device);
ENLSIPB200_API int enlsipb200_dense_mulq(int mr, int nq, int k, const double* f, const double* tau, double* M, int device);
/*   enlsipb200_dense_vecop : the vector products and triangular solves of src/enlsip_functions.jl:133-152, 484-500 as the
 *       engine runs them for long vectors (cooperative multi-CTA kernels).  kind 0: v [frows] <- Q' v, 1: v <- Q v with
 *       Q = H(0) ... H(k-1) from f [frows x k] / tau [k] (LAPACK dormqr); kind 2: v [k] <- R \ v, 3: v [k] <- R' \ v with
 *       R = the upper triangle of the leading k x k block of f [frows x k] (LAPACK dtrtrs).  Kinds 4-7: the operations of
 *       kinds 0-3 with the kernel the engine picks for that size (one warp, cooperative, or one CTA). */
ENLSIPB200_API int enlsipb200_dense_vecop(int kind, int frows, int k, const double* f, const double* tau, double* v, int device);
/*   enlsipb200_dense_gemv : the small stage's matrix-vector products.  A [rows x cols], leading dimension lda >= rows.
 *       trans 0: y [rows] = alpha A x + beta y0 (x [cols]; y0 [rows], NULL = 0); trans 1: y [cols] = A' x (x [rows];
 *       alpha, y0 and beta unused). */
ENLSIPB200_API int enlsipb200_dense_gemv(int trans, int rows, int cols, const double* A, int lda, const double* x, double alpha,
                                         const double* y0, double beta, double* y, int device);
/* device time (CUDA events around the kernels, transfers excluded) of the last enlsipb200_dense_* call, in ms */
ENLSIPB200_API float enlsipb200_dense_last_ms(void);

#ifdef __cplusplus
}
#endif
#endif
