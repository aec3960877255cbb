/* sqpb200.h -- C ABI of the B200-native batched QP-subproblem engine for RestartSQP.
 *
 * This is the drop-in boundary (SURVEY.md section 8b): what a `CudaQPInterface :
 * QPSolverInterface` adapter class (restartsqp_b200/csrc/adapter/CudaQPInterface.hpp) and the
 * batched host driver call.  No C++ types, no exceptions and no torch types cross this line.
 * Every function returns 0 on success, a negative SQPB200_ERR_* code on a library error, or,
 * for the solve status arrays, the reference's Exitflag QP codes 20..30
 * (include/sqphot/Types.hpp:51-73).
 *
 * One handle owns the device state of `batch` independent QP (or LP) instances that share
 * one sparsity pattern (one NLP structure), exactly the data one
 * `qpOASESInterface` object owns for a single instance (src/qpOASESInterface.cpp:106-128):
 * lb, ub, g, x [nV]; lbA, ubA [nC]; y [nV+nC]; A (CSC, nC x nV); H (CSC, nV x nV; QP only);
 * plus the hot-start state qpOASES keeps inside SQProblem (working set, TQ/Cholesky factors).
 *
 * Array arguments are caller-owned; `loc` says whether the pointer is host or device memory.
 * Batched arrays are instance-major: vals[batch][len], contiguous.
 * There is NO CPU fallback: every compute entry point runs CUDA kernels on the handle's device
 * and fails with SQPB200_ERR_CUDA if no device is available.
 */
#ifndef SQPB200_H
#define SQPB200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sqpb200_handle_s* sqpb200_handle;

#define SQPB200_LOC_HOST 0
#define SQPB200_LOC_DEVICE 1

/* QPType, include/sqphot/Types.hpp:45-48 */
#define SQPB200_LP 1
#define SQPB200_QP 2

/* vector selectors for sqpb200_set_vectors / get_vectors (setters at
 * include/sqphot/QPsolverInterface.hpp:144-165) */
#define SQPB200_VEC_G 0
#define SQPB200_VEC_LB 1
#define SQPB200_VEC_UB 2
#define SQPB200_VEC_LBA 3
#define SQPB200_VEC_UBA 4

#define SQPB200_MAT_A 0
#define SQPB200_MAT_H 1

/* ActiveType, include/sqphot/Types.hpp:84-89 */
#define SQPB200_ACTIVE_ABOVE 1
#define SQPB200_ACTIVE_BELOW (-1)
#define SQPB200_ACTIVE_BOTH_SIDE (-99)
#define SQPB200_INACTIVE 0

/* Exitflag QP codes, include/sqphot/Types.hpp:60-70 */
#define SQPB200_QP_OPTIMAL 20
#define SQPB200_QPERROR_INTERNAL_ERROR 21
#define SQPB200_QPERROR_INFEASIBLE 22
#define SQPB200_QPERROR_UNBOUNDED 23
#define SQPB200_QPERROR_EXCEED_MAX_ITER 24
#define SQPB200_QPERROR_NOTINITIALISED 25
#define SQPB200_QPERROR_PERFORMINGHOMOTOPY 28
#define SQPB200_QPERROR_UNKNOWN 30

#define SQPB200_ERR_INVALID (-1)
#define SQPB200_ERR_CUDA (-2)
#define SQPB200_ERR_NOMEM (-3)
#define SQPB200_ERR_STATE (-4)
#define SQPB200_ERR_TOO_LARGE (-5)

/* Solver options.  Defaults mirror Options::setToDefault (src/Options.cpp:19-57) for the
 * iteration limits and qpOASES Options::setToReliable (src/qpOASESInterface.cpp:765) for the rest. */
typedef struct {
    int qp_maxiter;      /* Options::qp_maxiter = 1000 */
    int lp_maxiter;      /* Options::lp_maxiter = 100 */
    int enable_flipping; /* 1 */
    int enable_ramping;  /* 1 */
    int enable_drift;    /* 1 */
    int team_size;       /* 0 = auto; 32 = one warp per QP (shared-memory resident); 1024 = one CTA per QP (slice in global memory, large QPs) */
    int keep_state;      /* 1: keep working set + factors resident for hot starts */
    int factor_cap;      /* capacity of the TQ/Cholesky factors = max. simultaneously free variables held in shared
                            memory: 0 = auto (n + m/2 + 2 for nV = n + 2m), -1 = nV.  Instances that need more are
                            re-solved with capacity nV by a rescue launch: the value affects speed, not results. */
    int debug_force_error_branch; /* test hook, 0 in production: every solve runs handle_error's infeasible branch after its first
                            attempt (re-init from the slack-feasible guess x0 = [0; max(0, lbA); -min(0, ubA)],
                            src/qpOASESInterface.cpp:716-729), which a feasible l1-penalty QP otherwise never reaches */
    int refactorise_every; /* one-QP-per-cluster kernel (team_size 1024) only.  0 (default): the projected Cholesky factor is carried
                            through an addition by rotations and recomputed every 64th addition; 1: recomputed after every
                            addition, as qpOASES does under setToReliable (enableCholeskyRefactorisation = 1) and as the warp
                            kernel always does.  Same matrix either way; O(nZ^2) against O(nZ^3) per working-set change. */
} sqpb200_options;

void sqpb200_default_options(sqpb200_options* o);
const char* sqpb200_version(void);
/* number of CUDA devices visible, or SQPB200_ERR_CUDA */
int sqpb200_device_count(void);

/* ---- life cycle: replaces qpOASESInterface ctor + allocate_memory (src/qpOASESInterface.cpp:35-50,
 * 106-128).  nV = nVar_QP, nC = nConstr_QP. */
int sqpb200_create(int batch, int nV, int nC, int qptype, int device, const sqpb200_options* opts,
                   sqpb200_handle* out);
int sqpb200_destroy(sqpb200_handle h);
/* run all subsequent work of this handle on the given cudaStream_t (NULL = default stream) */
int sqpb200_set_stream(sqpb200_handle h, void* cuda_stream);
int sqpb200_synchronize(sqpb200_handle h);
const char* sqpb200_last_error(sqpb200_handle h);

/* ---- structure: replaces set_A / set_H first call -> SpHbMat::setStructure
 * (src/qpOASESInterface.cpp:426-437, 400-417; src/SpHbMat.cpp:196-268, 284-355).
 * Triplets are 1-based (FORTRAN style, src/SQPTNLP.cpp:18).  The identity blocks are the
 * IdentityInfo of include/sqphot/Types.hpp:36-42.  Runs the device segmented sort/scan.
 * Returns the number of CSC entries (>= 0) or a negative error. */
int sqpb200_set_structure_A(sqpb200_handle h, int zJ, const int* row1, const int* col1, int I_len,
                            const int* I_irow, const int* I_jcol, const int* I_size,
                            const double* I_value);
int sqpb200_set_structure_H(sqpb200_handle h, int zH, const int* row1, const int* col1,
                            int is_symmetric);
/* Direct CSC structure (the data constructor used by the replay driver,
 * src/qpOASESInterface.cpp:54-94, test/QPsolvers_testers.cpp:220-221). */
int sqpb200_set_structure_csc(sqpb200_handle h, int which, int nnz, const int* colptr,
                              const int* rowidx);
/* Copy the CSC index arrays back to the host for parity checks: colptr[ncol+1], rowidx[nnz],
 * order[nnz] (order may be NULL). */
int sqpb200_get_structure(sqpb200_handle h, int which, int* colptr, int* rowidx, int* order);
int sqpb200_get_nnz(sqpb200_handle h, int which);

/* ---- values: replaces set_A / set_H later calls -> SpHbMat::setMatVal (src/SpHbMat.cpp:368-393).
 * vals[batch][z] are triplet-ordered values (zJ per instance for A, zH for H); they are scattered
 * through `order` on the device.  broadcast != 0: vals[z] is shared by all instances. */
int sqpb200_set_values_A(sqpb200_handle h, const double* vals, int loc, int broadcast);
int sqpb200_set_values_H(sqpb200_handle h, const double* vals, int loc, int broadcast);
/* CSC-ordered values (data-constructor path). */
int sqpb200_set_values_csc(sqpb200_handle h, int which, const double* vals, int loc, int broadcast);
int sqpb200_get_values_csc(sqpb200_handle h, int which, double* vals, int loc);

/* ---- vectors: bulk form of set_lb/set_ub/set_lbA/set_ubA/set_g
 * (src/qpOASESInterface.cpp:361-395, 445-484).  Writes vals[batch][count] into entries
 * [offset, offset+count) of the selected vector of every instance and raises the same change
 * flags (Update_bounds / Update_g).  broadcast != 0: vals[count] shared by all instances. */
int sqpb200_set_vectors(sqpb200_handle h, int which, const double* vals, int offset, int count,
                        int loc, int broadcast);
int sqpb200_get_vectors(sqpb200_handle h, int which, double* vals, int loc);

/* ---- batched QPhandler data construction on the device (src/QPhandler.cpp:167-261, 272-297,
 * 342-419, 430-463, 533-567): n = NLP variables, m = NLP constraints (nV = n+2m, nC = m).
 * mode 0 = set_bounds, 1 = update_bounds as the reference's non-QORE branch does it (lbA refreshed, ubA left stale:
 * src/QPhandler.cpp:358-360), 2 = update_delta, 3 = update_bounds refreshing lbA and ubA (what the QORE branch does, :377-382).
 * delta[batch]; x_l,x_u,x_k [batch][n]; c_l,c_u,c_k [batch][m] (device or host per loc). */
int sqpb200_qphandler_bounds(sqpb200_handle h, int mode, int n, int m, const double* delta,
                             const double* x_l, const double* x_u, const double* x_k,
                             const double* c_l, const double* c_u, const double* c_k, int loc);
/* g = [grad ; rho*1]: grad[batch][n] may be NULL (update_penalty), rho[batch] may be NULL
 * (update_grad). */
int sqpb200_qphandler_g(sqpb200_handle h, int n, int m, const double* grad, const double* rho,
                        int loc);

/* ---- solve: replaces optimizeQP / optimizeLP incl. the init/hotstart state machine and the
 * one-retry recovery (src/qpOASESInterface.cpp:137-284, 686-758, 817-833).
 * mode = SQPB200_QP or SQPB200_LP; maxiter <= 0 uses the option default; active_mask[batch]
 * (host, may be NULL = all) selects the instances to solve. */
int sqpb200_solve(sqpb200_handle h, int mode, int maxiter, const unsigned char* active_mask);

/* ---- one call per solve for host-resident data (the end-to-end path of a host driver that keeps a pinned mirror of the handle's
 * data; replaces the per-entry setters + optimizeQP + getters of src/qpOASESInterface.cpp:137-224, 290-357, 361-484 for a whole
 * batch).  sqpb200_io_layout gives the layout of the handle's two contiguous blocks: in_off5 = byte offsets of g, lb, ub, lbA,
 * ubA ([batch][len] each) inside the input block of in_bytes bytes; out_off6 = byte offsets of x, y, obj, kkt[5], status (int32),
 * iters (int32) inside the result block of out_bytes bytes.  sqpb200_solve_host queues: one host-to-device copy of the input
 * block (NULL: unchanged), one each of the CSC-ordered A / H values [batch][nnz] (NULL: unchanged; raises Update_A / Update_H),
 * the solve, and one device-to-host copy of the result block (NULL: skipped).  Nothing is waited for: sqpb200_synchronize. */
int sqpb200_io_layout(sqpb200_handle h, size_t* in_off5, size_t* in_bytes, size_t* out_off6, size_t* out_bytes);
int sqpb200_solve_host(sqpb200_handle h, int mode, int maxiter, const void* in_block, const double* Aval_csc,
                       const double* Hval_csc, void* out_block);

/* ---- results (src/qpOASESInterface.cpp:221-222, 290-357).  Any pointer may be NULL.
 * x[batch][nV]; y[batch][nV+nC] (bound multipliers first); obj[batch]; status[batch] (Exitflag);
 * iters[batch] (working-set changes of the last solve, what the reference adds to Stats::qp_iter). */
int sqpb200_get_solution(sqpb200_handle h, double* x, double* y, double* obj, int* status,
                         int* iters, int loc);
/* wb[batch][nV], wc[batch][nC] as int32.  translated = 0: raw qpOASES convention (+1 upper,
 * -1 lower, 0 inactive); translated = 1: the reference's ActiveType after get_working_set
 * (src/qpOASESInterface.cpp:835-895). */
int sqpb200_get_working_set(sqpb200_handle h, int* wb, int* wc, int translated, int loc);
/* out[batch][5] = primal, dual, stationarity, complementarity violation and KKT_error of
 * test_optimality (src/qpOASESInterface.cpp:498-684), evaluated by the solve kernel's epilogue. */
int sqpb200_kkt_residuals(sqpb200_handle h, double* out, int loc);
/* Recompute them with the stand-alone batched kernel (for parity tests and ncu). */
int sqpb200_kkt_residuals_recompute(sqpb200_handle h, double* out, int loc);

/* ---- stand-alone batched SpMV / SpMTV on the handle's CSC matrices (SpHbMat::times,
 * transposed_times; src/SpHbMat.cpp:659-737).  x[batch][ncol or nrow], y[batch][nrow or ncol]. */
int sqpb200_spmv(sqpb200_handle h, int which, int transpose, const double* x, double* y, int loc);

/* ---- batched Vector operations (row A2 of SURVEY.md 8a: src/Vector.cpp:94-135, 174-184, 237-251; Utils oneNorm / infNorm,
 * src/Utils.cpp:65-83) on [batch][n] arrays, no handle needed.  Reductions sum in the reference's index order per instance, so
 * results are bit-identical with Vector::getOneNorm / getInfNorm / times.
 * sqpb200_vector_reduce: op 0 = getOneNorm, 1 = getInfNorm, 2 = times (dot product with y); out[batch].
 * sqpb200_vector_elementwise (in place on x): op 0 = add_vector (x += y), 1 = subtract_vector (x -= y), 2 = subtract_vector_to
 * (x = y - x), 3 = addNumber (x += alpha), 4 = copy_vector (x = y), 5 = scale (x *= alpha). */
int sqpb200_vector_reduce(int device, int op, long long batch, int n, const double* x, const double* y, double* out, int loc,
                          void* stream);
int sqpb200_vector_elementwise(int device, int op, long long batch, int n, double* x, const double* y, double alpha, int loc,
                               void* stream);

/* ---- stand-alone segmented triplet -> CSC assembly over `nmat` independent matrices in one
 * launch (rows A4/A5 as a batched device sort/scan).  seg[nmat+1] are offsets into the 1-based
 * triplet arrays; ncol[nmat] column counts.  Outputs: colptr (concatenated, sum(ncol+1)),
 * rowidx and order (same offsets as the input).  All pointers host memory. */
int sqpb200_assemble_csc_batched(int device, int nmat, const int* seg, const int* ncol,
                                 const int* row1, const int* col1, int* colptr, int* rowidx,
                                 int* order, float* kernel_ms);

/* kernels launched by this handle since creation (for bench.py's gpu_launches) */
long long sqpb200_launch_count(sqpb200_handle h);
/* Developer aid: cycle counters per solver phase, summed over all instances since the last reset (out16[16]; all zero unless the
 * library was built with SQPB200_QP_FLAGS=-DQP_PROFILE; indices = the PR_* enum of csrc/qp_kernel.cuh). */
int sqpb200_get_profile(sqpb200_handle h, long long* out16, int reset);
/* smem bytes per QP, team size and QPs per CTA chosen for the solve kernel */
int sqpb200_solve_config(sqpb200_handle h, int* team_size, int* qps_per_cta, int* smem_per_cta);
/* device time of the last solve launch measured with CUDA events on the handle's stream (ms) */
float sqpb200_last_solve_ms(sqpb200_handle h);

/* ---- batched NLP evaluation on the device (the step on the other side of the path: what the reference gets from
 * Ipopt's AmplTNLP through SQPTNLP::Eval_f / Eval_gradient / Eval_constraints / Eval_Jacobian / Eval_Hessian,
 * src/SQPTNLP.cpp:67-132).  `cuda_source` defines two kernels, one thread per instance:
 *   nlp_eval_fc (int B, const double* x, double* f, double* c)
 *   nlp_eval_all(int B, const double* x, const double* lam, double* f, double* c, double* grad, double* jac, double* hess)
 * (x[B][n], lam[B][m], c[B][m], grad[B][n], jac[B][zJ], hess[B][zH]); it is compiled with NVRTC for sm_100a
 * (--fmad=false).  compile needs no GPU; load / eval do and fail with SQPB200_ERR_CUDA without one. */
typedef struct sqpb200_nlp_s* sqpb200_nlp;
int sqpb200_nlp_compile(const char* cuda_source, int n, int m, int zJ, int zH, char* log, int log_len, sqpb200_nlp* out);
long long sqpb200_nlp_cubin_size(sqpb200_nlp h);
int sqpb200_nlp_load(sqpb200_nlp h, int device);
/* which = 0: f and c; 1: f, c, grad, jac, hess (lam = the multipliers the caller wants in the Lagrangian Hessian:
 * Algorithm passes -lambda, src/SQPTNLP.cpp:124-126).  NULL outputs are skipped; loc as everywhere. */
int sqpb200_nlp_eval(sqpb200_nlp h, int which, int B, const double* x, const double* lam, double* f, double* c,
                     double* grad, double* jac, double* hess, int loc, void* stream);
int sqpb200_nlp_destroy(sqpb200_nlp h);
long long sqpb200_nlp_launch_count(sqpb200_nlp h);
const char* sqpb200_nlp_last_error(void);

/* ---- device-resident outer loop (SURVEY.md 8f-1): the per-instance steps of Algorithm::Optimize (src/Algorithm.cpp:55-168)
 * as phases of one kernel, one thread per instance, over SoA state that never leaves the device.  The caller owns every
 * array (device memory) and sequences phases, QP/LP solves (sqpb200_solve_device_mask) and NLP evaluations (sqpb200_nlp_eval
 * with device pointers). */
/* exit flag of an instance whose QP data did not change since its last solve (no Update_* flag raised): the reference's setupQP
 * throws QP_UNCHANGED there (src/Algorithm.cpp:651-670) and nothing catches it; 7 is not a value of the reference's Exitflag */
#define SQPB200_EXIT_QP_UNCHANGED 7
#define SQPB200_PH_FLAGS 0
#define SQPB200_PH_AFTER_QP 1
#define SQPB200_PH_LP_AFTER 2
#define SQPB200_PH_PEN_CHECK 3
#define SQPB200_PH_PEN_AFTER 4
#define SQPB200_PH_PEN_FINAL 5
#define SQPB200_PH_TRIAL 6
#define SQPB200_PH_RATIO 7
#define SQPB200_PH_FINISH 8
#define SQPB200_PH_FINAL 9
#define SQPB200_PH_SOC_PREP 10
#define SQPB200_PH_SOC_AFTER 11
#define SQPB200_PH_SOC_RATIO 12
#define SQPB200_PH_INIT 13
typedef struct {
    int B, n, m, zJ, zH;
    /* Options (src/Options.cpp:19-57) */
    int iter_max, penalty_update, penalty_iter_max, clear_flags;
    double eta_c, eta_s, eta_e, gamma_c, gamma_e, delta_min, delta_max, tol, penalty_update_tol, rho_max, increase_parm,
        eps1_change_parm, eps2, opt_prim_fea_tol, opt_dual_fea_tol, opt_compl_tol, opt_stat_tol;
    /* model: Jacobian triplet pattern (1-based), bounds and constraint classes per instance */
    const int *J_row1, *J_col1;
    const double *x_l, *x_u, *c_l, *c_u;      /* [B][n], [B][m] */
    const int *bound_type, *cons_type;        /* ConstraintType, include/sqphot/Types.hpp:75-81 */
    /* iterate and algorithm state, [B][...] */
    double *x_k, *c_k, *f_k, *grad, *jac, *hess, *lam_c, *lam_x, *neg_lam;
    double *delta, *rho, *eps1, *infea, *p_k, *x_trial, *c_trial, *f_trial, *infea_trial, *infea_model, *infea_model_tmp,
        *rho_trial, *infea_infty, *actual_red, *pred_red, *kkt_err;
    double *g_new, *j_new, *h_new;            /* derivatives at the trial point of accepted steps */
    double* scratch;                          /* [B][n] */
    int *exitflag, *iter, *pen_trial;
    long long* qp_iter;
    unsigned char *active, *need, *go, *acc, *upd, *feasible_lp;
    /* result buffers of the QP and LP handles (sqpb200_device_buffers) */
    const double *qp_x, *qp_y, *qp_obj, *qp_kkt, *lp_x;
    const int *qp_status, *qp_iters, *lp_status, *lp_iters;
    int* counters;                            /* [8] device */
    /* second-order correction (src/Algorithm.cpp:1140-1211, opt-in): Hessian triplet pattern, mixed QP data, saved step */
    const int *H_row1, *H_col1;
    double *soc_g, *soc_x, *soc_c, *p_tmp, *qp_obj_tmp, *qp_obj_soc, *norm_p;
    unsigned char* rej;
    /* per-instance backend state machines of the QP and the LP handle (sqpb200_solve_per_instance); NULL: handle-level modes */
    signed char *qp_inst, *lp_inst;
    /* start values of delta, rho, eps1 (Options, src/Options.cpp:19-57), applied by SQPB200_PH_INIT */
    double delta0, rho0, eps10;
} sqpb200_sqp_state;
/* counters_host (may be NULL): the 8 device counters after the phase ([0] active instances, [1] OR of the raised Update_*
 * bits 1=A 2=H 4=bounds 8=delta 16=penalty 32=g, [2] instances needing the penalty update, [3] instances continuing the
 * penalty loop, [4] accepted steps, [5] rejected steps entering the second-order correction); reading them synchronises the
 * stream. */
int sqpb200_sqp_phase(const sqpb200_sqp_state* st, int phase, int* counters_host, void* stream);
/* The whole of Algorithm::Optimize (src/Algorithm.cpp:55-168) for the batch: phases, QP data updates (setupQP :645-697), QP / LP
 * solves (update_penalty_parameter :886-1028), NLP evaluations and, if requested, the second-order correction (:1140-1211),
 * sequenced from C++ on `stream` (which must be the stream of both handles).  The caller has set the structures of both handles
 * and evaluated f, c, grad, jac, hess at the start point; *first (in/out) is 1 before the first outer iteration; f_tmp[B] and
 * c_tmp[B][m] receive the function values of the derivative evaluation (unused by the algorithm).  refresh_ubA: 1 = update_bounds
 * refreshes both constraint sides (mode 3 of sqpb200_qphandler_bounds), 0 = the reference's stale-ubA behaviour (mode 1). */
int sqpb200_sqp_optimize(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp, int second_order_correction,
                         int refresh_ubA, int* first, double* f_tmp, double* c_tmp, long long* launches, void* stream);
/* Streamed solves: N starting points through the B = st->B instances ("slots") of the state.  A slot whose instance has stopped
 * hands its results to out[instance] and takes the next starting point of the queue, so the batch does not wait for its slowest
 * instance.  Every array is device memory owned by the caller; the function sets slot_id to -1, *head to 0 and refill to 0 itself. */
typedef struct {
    long long N;              /* number of starting points */
    int refill_min;           /* a refill round runs once at least this many occupied slots have stopped (>= 1), or when none is active */
    const double* x0_all;     /* [N][n] starting points (shifted into the bounds as initialization() does) */
    const double* lam_start;  /* [m] starting constraint multipliers (NULL if m = 0) */
    /* results by instance (input order): final iterate, objective, exit flag (as sqpb200_sqp_optimize leaves them), outer and QP
     * iterations, KKT error, penalty parameter, trust-region radius */
    double* x;                /* [N][n] */
    double *obj, *kkt_err, *rho, *delta;
    int *exitflag, *iter;
    long long* qp_iter;
    long long* slot_id;       /* [B] instance held by each slot, -1 = free */
    unsigned long long* head; /* [1] next queue index (advanced with atomicAdd; may end above N) */
    unsigned char* refill;    /* [B] slots filled by the last refill round */
    long long rounds;         /* out: refill rounds, the initial fill included */
} sqpb200_sqp_stream;
/* Algorithm::Optimize for every starting point of `sd`, same arguments as sqpb200_sqp_optimize otherwise.  Each instance follows
 * exactly the trajectory it follows in one batch with all N (instances do not influence each other).  Needs per-instance backend
 * state machines (st->qp_inst and st->lp_inst set): with handle-level modes the instances of a handle share its init / hotstart
 * decision, so SQPB200_ERR_INVALID.  Returns when the queue is empty and every instance has been collected; the state's own
 * per-instance arrays then hold the slots' last instances. */
int sqpb200_sqp_optimize_stream(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp,
                                int second_order_correction, int refresh_ubA, int* first, double* f_tmp, double* c_tmp,
                                sqpb200_sqp_stream* sd, long long* launches, void* stream);
/* Asynchronous solves: the loop of sqpb200_sqp_optimize recorded once as a CUDA graph whose branches (does any instance remain
 * active, need the penalty update, continue the penalty loop, enter the second-order correction, is a refill round due) are
 * conditional nodes set on the device from the counters.  A launch queues the whole solve on `stream` and returns: nothing is read
 * back and nothing is waited for, so solves of several states can run concurrently on several streams from one host thread.
 * Results are bit-identical with the synchronous calls for the same sequence of calls on a state.
 *
 * sqpb200_sqp_graph_create: same preconditions and arguments as sqpb200_sqp_optimize (structures set, start evaluated; `stream` is
 * the stream of both handles), plus per-instance backend state machines (st->qp_inst and st->lp_inst), else SQPB200_ERR_INVALID.
 * It makes the handles' first-solve allocations and records the loop (synchronising nothing).  `st` is kept by pointer: it and every
 * array it names must stay valid and unchanged, except clear_flags, until sqpb200_sqp_graph_destroy; the handles' stream too.
 * sqpb200_sqp_graph_launch: sd == NULL queues one sqpb200_sqp_optimize; sd != NULL one sqpb200_sqp_optimize_stream over the
 * descriptor (recording its loop again, since the descriptor is part of the graph: the launch then costs a capture and an
 * instantiation).  *first as in those calls, updated when the launch is queued; sd->rounds and launch counts are not reported.
 * The results are in place once the stream reaches them (an event recorded after the launch).
 * sqpb200_sqp_graph_destroy: a graph still running is released when it completes. */
typedef struct sqpb200_sqp_graph_s* sqpb200_sqp_graph;
int sqpb200_sqp_graph_create(sqpb200_sqp_state* st, sqpb200_handle qp, sqpb200_handle lp, sqpb200_nlp nlp, int second_order_correction,
                             int refresh_ubA, double* f_tmp, double* c_tmp, void* stream, sqpb200_sqp_graph* out);
int sqpb200_sqp_graph_launch(sqpb200_sqp_graph g, int* first, sqpb200_sqp_stream* sd);
int sqpb200_sqp_graph_destroy(sqpb200_sqp_graph g);
/* Forget every solve so far: the next solve is an init (cold start) again, as for a freshly constructed backend
 * (firstQPsolved_ = false, matrix status UNDEFINED, Update_* flags cleared; src/qpOASESInterface.cpp:35-50).  Structures and
 * device buffers are kept, so one handle can serve batch after batch. */
int sqpb200_reset(sqpb200_handle h);
/* sqpb200_solve with the instance mask in device memory */
int sqpb200_solve_device_mask(sqpb200_handle h, int mode, int maxiter, const unsigned char* device_mask);
/* The same with the init / hotstart decision (src/qpOASESInterface.cpp:141-211, 817-833) made PER INSTANCE inside the kernel, as the
 * reference does for its single instance: inst_state[batch][8] (int8, device memory, owned by the caller, initialised to
 * {0, 0, -1, -1, 0, ...}) holds {first_solved, varied, old matrix status, new matrix status, last mode}; the caller sets
 * varied = 1 for an instance whenever it hands that instance new matrix values (csrc/sqp_outer.cu does).  Needs keep_state. */
int sqpb200_solve_per_instance(sqpb200_handle h, int mode, int maxiter, const unsigned char* device_mask,
                               signed char* device_inst_state);
/* device pointers of the handle's result arrays: out[0..5] = x, y, obj, status, iters, kkt */
int sqpb200_device_buffers(sqpb200_handle h, void** out);

/* ---- QORE layout (SURVEY.md 8f rank 4): the wire format of the reference's QORE backend -- compressed-row matrices and bounds
 * stacked as lb = [lb_x ; lb_Ax], ub = [ub_x ; ub_Ax] of length nV + nC (include/sqphot/QOREInterface.hpp:30-252;
 * src/QOREInterface.cpp:89-90 QPSetData(A_->RowIndex(), A_->ColIndex(), A_->MatVal(), H_->...), :102 QPOptimize(lb_, ub_, g_),
 * :120-122 "primalsol" / "dualsol" of length nV + nC, :441 "workingset"; the QPhandler side is src/QPhandler.cpp:225-260,
 * 369-383).  A handle whose structure was given this way solves on the same kernels: the column-compressed pattern the solver
 * works on is derived once, values move through a precomputed position map on the device.
 *
 * sqpb200_set_structure_A_csr / _H_csr: first call of QOREInterface::set_A / set_H (src/QOREInterface.cpp:643-659) ->
 * SpHbMat(..., isCompressedRow = true)::setStructure (src/SpHbMat.cpp:238-250, 324-337): same arguments as
 * sqpb200_set_structure_A / _H, same device sort with the key (row, column, counter); later sqpb200_set_values_A / _H calls take
 * triplet-ordered values as before.  Return the number of entries or a negative error. */
int sqpb200_set_structure_A_csr(sqpb200_handle h, int zJ, const int* row1, const int* col1, int I_len,
                                const int* I_irow, const int* I_jcol, const int* I_size, const double* I_value);
int sqpb200_set_structure_H_csr(sqpb200_handle h, int zH, const int* row1, const int* col1, int is_symmetric);
/* Direct compressed-row structure: the data constructor QOREInterface(H, A, g, lb, ub, options) of the replay driver
 * (src/QOREInterface.cpp:36-60, test/QPsolvers_testers.cpp:74-75, 172-175).  rowptr[nrow+1], colidx[nnz], 0-based, entries of a
 * row in ascending column order.  Values then arrive in this storage order through sqpb200_set_values_csr. */
int sqpb200_set_structure_csr(sqpb200_handle h, int which, int nnz, const int* rowptr, const int* colidx);
/* rowptr[nrow+1], colidx[nnz], order[nnz] (triplet entry -> storage position; any pointer may be NULL) of a handle whose
 * structure was set through one of the three calls above. */
int sqpb200_get_structure_csr(sqpb200_handle h, int which, int* rowptr, int* colidx, int* order);
/* vals[batch][nnz] in compressed-row storage order (broadcast != 0: vals[nnz] shared by all instances); raises Update_A / Update_H
 * like QOREInterface::set_A / set_H (matrix_change_flag_, src/QOREInterface.cpp:647, 656). */
int sqpb200_set_values_csr(sqpb200_handle h, int which, const double* vals, int loc, int broadcast);
int sqpb200_get_values_csr(sqpb200_handle h, int which, double* vals, int loc);
/* Stacked bounds lb[batch][nV+nC], ub[batch][nV+nC] (either may be NULL): bulk form of QOREInterface::set_lb / set_ub
 * (include/sqphot/QOREInterface.hpp; written by src/QPhandler.cpp:225-260, 369-383).  Entries [0, nV) are the variable bounds,
 * [nV, nV+nC) the constraint bounds.  broadcast != 0: one row shared by all instances. */
int sqpb200_set_bounds_stacked(sqpb200_handle h, const double* lb, const double* ub, int loc, int broadcast);
int sqpb200_get_bounds_stacked(sqpb200_handle h, double* lb, double* ub, int loc);
/* Results in QORE's layout (src/QOREInterface.cpp:120-122, 441): primal[batch][nV+nC] = [x ; A x], dual[batch][nV+nC] = [bound
 * multipliers ; constraint multipliers], workingset[batch][nV+nC] (int32) in QORE's sign convention as the reference decodes it
 * (src/QOREInterface.cpp:440-492: -1 = active at the upper bound, +1 = active at the lower bound, 0 = inactive).  Any pointer
 * may be NULL. */
int sqpb200_get_solution_stacked(sqpb200_handle h, double* primal, double* dual, int* workingset, int loc);

#ifdef __cplusplus
}
#endif
#endif /* SQPB200_H */
