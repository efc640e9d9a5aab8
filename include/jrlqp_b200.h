/* jrlqp_b200.h — C-ABI of the B200-native batched Goldfarb-Idnani QP solver.
 *
 * Drop-in boundary for ONE path of jrl-umi3218/jrl-qp: GoldfarbIdnaniSolver::solve
 * (include/jrl-qp/GoldfarbIdnaniSolver.h:27-33, src/GoldfarbIdnaniSolver.cpp:18-54) and the
 * DualSolver accessors (include/jrl-qp/DualSolver.h:26-60), batched: every call solves `batch`
 * independent strictly convex QPs
 *
 *      min 1/2 x^T G x + a^T x   s.t.  bl <= C^T x <= bu,  xl <= x <= xu
 *
 * with hand-written FP64 CUDA kernels for sm_100a. batch == 1 behaves like one call on the
 * reference object. The reference has no FFI layer of its own (it is a C++ class library over
 * Eigen::Ref views); the entry points below carry exactly what those views carry: a pointer, a
 * leading dimension, and — because the call is batched — an element stride between instances
 * (0 = the array is shared by all instances).
 *
 * There is no CPU fallback: every entry point fails with JRLQP_ERR_CUDA when no sm_100 device
 * is usable.
 *
 * Plain C: pointers, sizes and PODs only (no torch / Eigen / STL types).
 */
#ifndef JRLQP_B200_H
#define JRLQP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C"
{
#endif

#define JRLQP_B200_VERSION 200 /* 0.2.0: multi-GPU entry points, one in-flight device call per handle */

/* include/jrl-qp/enums.h:14-23 — jrl::qp::ActivationStatus (same values, int8 storage) */
enum jrlqp_activation_status
{
  JRLQP_INACTIVE = 0,
  JRLQP_LOWER = 1,
  JRLQP_UPPER = 2,
  JRLQP_EQUALITY = 3,
  JRLQP_LOWER_BOUND = 4,
  JRLQP_UPPER_BOUND = 5,
  JRLQP_FIXED = 6
};

/* include/jrl-qp/enums.h:26-37 — jrl::qp::TerminationStatus (same values) */
enum jrlqp_termination_status
{
  JRLQP_SUCCESS = 0,
  JRLQP_INCONSISTENT_INPUT = 1,
  JRLQP_NON_POS_HESSIAN = 2,
  JRLQP_INFEASIBLE = 3,
  JRLQP_MAX_ITER_REACHED = 4,
  JRLQP_LINEAR_DEPENDENCY_DETECTED = 5,
  JRLQP_OVERCONSTRAINED_PROBLEM = 6,
  JRLQP_UNKNOWN = 7
};

/* Library-level error codes (returned by the API functions; never stored in status arrays). */
#define JRLQP_OK 0
#define JRLQP_ERR_CUDA (-1) /* CUDA runtime/driver error, or no sm_100 device */
#define JRLQP_ERR_ARG (-2) /* invalid argument (sizes, null pointer, unsupported n) */
#define JRLQP_ERR_CAPACITY (-3) /* batch larger than the capacity given to jrlqp_create */

/* include/jrl-qp/SolverOptions.h:14-22 — jrl::qp::SolverOptions. log_flags is carried for API
 * parity only: the Matlab-syntax logger (include/jrl-qp/utils/Logger.h) is out of scope. */
typedef struct jrlqp_options
{
  int32_t max_iter; /* maxIter_  = 500   */
  double big_bnd; /* bigBnd_   = 1e100 */
  int32_t warm_start; /* warmStart_ = false; honoured only by jrlqp_solve_batch_warm_* */
  uint32_t log_flags; /* logFlags_ = 0     */
} jrlqp_options;

/* One batch of problems. All pointers live in the same memory space (device for *_device entry
 * points, host for *_host). "stride" = distance in ELEMENTS between instance k and k+1; 0 shares
 * the array. Matrices are column-major with a leading dimension, as Eigen::Ref<MatrixXd> views
 * (include/jrl-qp/defs.h:11-14).
 *   G  n x n, lower triangle read (src/GoldfarbIdnaniSolver.cpp:58). NOT overwritten: the factor
 *      the reference leaves in G is returned through jrlqp_result.L when asked for.
 *   C  n x mc, one constraint normal per column (include/jrl-qp/GoldfarbIdnaniSolver.h:22-26).
 *   xl == NULL  <=>  no bounds (src/GoldfarbIdnaniSolver.cpp:28).
 *   as_in: optional warm-start activation status, int8 x (mc+nb) per instance, general
 *      constraints first (include/jrl-qp/experimental/GoldfarbIdnaniSolver.h:27-34).
 */
typedef struct jrlqp_problem
{
  int64_t batch;
  const double * G;
  int64_t G_stride;
  int32_t ldg;
  const double * a;
  int64_t a_stride;
  const double * C;
  int64_t C_stride;
  int32_t ldc;
  const double * bl;
  int64_t bl_stride;
  const double * bu;
  int64_t bu_stride;
  const double * xl;
  int64_t xl_stride;
  const double * xu;
  int64_t xu_stride;
  const int8_t * as_in;
  int64_t as_stride;
} jrlqp_problem;

/* Dense outputs, instance-major. Any pointer may be NULL (that output is skipped) except x.
 *   x           [batch][n]        DualSolver::solution()       src/DualSolver.cpp:33-36
 *   u           [batch][mc+nb]    DualSolver::multipliers()    src/DualSolver.cpp:38-69 (signed,
 *                                 + for UPPER/UPPER_BOUND, - otherwise; constraints then bounds)
 *   f           [batch]           DualSolver::objectiveValue() src/DualSolver.cpp:71-74
 *   iterations  [batch]           DualSolver::iterations()     src/DualSolver.cpp:76-79
 *   status      [batch]           return value of solve()      (jrlqp_termination_status)
 *   active_set  [batch][mc+nb]    DualSolver::activeSet()      (jrlqp_activation_status, int8)
 *   active_list [batch][n]        ordered active list (ActiveSet::operator[]), -1 padded
 *   n_active    [batch]           ActiveSet::nbActiveCstr()
 *   L           [batch][n][n]     column-major, ld n: lower triangle = Cholesky factor that the
 *                                 reference leaves in G (strict upper triangle not written)
 * On JRLQP_NON_POS_HESSIAN x, u, f are zero and the active set is empty (the reference leaves
 * them unspecified).
 */
typedef struct jrlqp_result
{
  double * x;
  double * u;
  double * f;
  int32_t * iterations;
  int32_t * status;
  int8_t * active_set;
  int32_t * active_list;
  int32_t * n_active;
  double * L;
} jrlqp_result;

typedef struct jrlqp_solver jrlqp_solver;

/* GoldfarbIdnaniSolver(nbVar, nbCstr, useBounds) (include/jrl-qp/GoldfarbIdnaniSolver.h:17-19)
 * + DualSolver::resize. batch_capacity bounds the batch of the *_host entry points (device staging
 * buffers are allocated once here, honouring the reference's no-allocation-in-solve contract,
 * tests/GoldfarbIdnaniSolverTest.cpp:113-117). device = CUDA ordinal. n <= 1024: problems with
 * n <= 128 keep J and R in shared memory for the whole solve; larger ones (the reference's MultiIK
 * fixtures, n = 387 / 210) use a per-CTA workspace in global memory (L2-resident). */
int jrlqp_create(jrlqp_solver ** out, int32_t n, int32_t mc, int32_t use_bounds, int64_t batch_capacity, int32_t device);
int jrlqp_destroy(jrlqp_solver * s);

/* DualSolver::options(const SolverOptions&) (src/DualSolver.cpp:26-31) */
void jrlqp_default_options(jrlqp_options * opt);
int jrlqp_set_options(jrlqp_solver * s, const jrlqp_options * opt);
int jrlqp_get_options(const jrlqp_solver * s, jrlqp_options * opt);

/* GoldfarbIdnaniSolver::solve (src/GoldfarbIdnaniSolver.cpp:18-54), batched, DEVICE pointers,
 * asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream).
 * Returns JRLQP_OK once enqueued; per-instance statuses land in res->status.
 * One call in flight per HANDLE: a solver owns single-buffered device scratch (as the reference's solver object owns
 * its workspaces, src/DualSolver.cpp:251-274), so a call enqueued on another stream than the previous one first waits
 * for it on the device (event). Use one handle per stream for concurrent batches. */
int jrlqp_solve_batch_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, void * stream);

/* Same call with HOST pointers: host->device copies, the kernels, device->host copies, then a
 * synchronise. Host memory may be pageable or pinned. Returns the worst jrlqp_termination_status
 * of the batch (>= 0) or a negative JRLQP_ERR_*. */
int jrlqp_solve_batch_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res);

/* experimental::GoldfarbIdnaniSolver::solve(G, a, C, bl, bu, xl, xu, as)
 * (include/jrl-qp/experimental/GoldfarbIdnaniSolver.h:27-34, src/experimental/GoldfarbIdnaniSolver.cpp:21-111,
 * 306-486), the warm-start capable solver, batched: the guessed active set pb->as_in (nullable) is
 * honoured when options.warm_start != 0 — equalities of the data always are —, the corresponding
 * normals are factorised at once (B = L^-1 N = Q R, J = L^-T Q), constraints that come out with a
 * negative multiplier are dropped, and the usual iteration follows; `iterations` counts those drops
 * plus the iterations, so a correct guess gives 0 (tests/GoldfarbIdnaniSolverTest.cpp:176-181).
 * The reference's "as empty => reuse the active set of the previous call" is the caller passing the
 * previous result's active_set back as as_in. Guesses that cannot apply are ignored as in the
 * reference (FIXED on distinct bounds, a side whose bound is infinite); statuses of the wrong kind
 * (a bound status on a general constraint or vice versa), on which the reference asserts, are ignored.
 * JRLQP_OVERCONSTRAINED_PROBLEM is reported per instance when more than n equalities are given.
 * The shared-memory kernel needs n (n - 1) / 2 more doubles of shared memory than the cold one, so it
 * fits up to n = 115 or so (the limit depends slightly on mc). In automatic mode a warm call whose layout
 * does not fit runs on the global-workspace kernel (bit-identical results) while cold calls on the same
 * handle keep the shared-memory kernel; with jrlqp_set_kernel_path(1) it returns JRLQP_ERR_ARG. */
int jrlqp_solve_batch_warm_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, void * stream);
int jrlqp_solve_batch_warm_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res);

/* Introspection used by the benchmark harness. */
typedef struct jrlqp_kernel_info
{
  int32_t threads_per_qp; /* 32 * warps: one QP per CTA */
  int32_t rows_per_thread;
  int32_t smem_bytes_per_qp;
  int32_t qps_per_sm; /* resident CTAs per SM */
  int32_t grid; /* persistent CTAs */
  int32_t num_sms;
  int32_t stage_c; /* 1: constraint matrix staged in shared memory */
  int32_t regs_per_thread;
} jrlqp_kernel_info;
int jrlqp_get_kernel_info(const jrlqp_solver * s, jrlqp_kernel_info * info);
/* Tuning knob: 0 = C read from global/L2, 1 = staged in shared memory, -1 = automatic. */
int jrlqp_set_stage_c(jrlqp_solver * s, int32_t mode);
/* Kernel family: 0 = automatic (n <= 128: shared-memory kernel, else global-workspace kernel),
 * 1 = shared-memory kernel (n <= 128), 2 = global-workspace kernel (any n <= 1024; used by the tests
 * to cross-check the two families on the same problems — their results are bit-identical). */
int jrlqp_set_kernel_path(jrlqp_solver * s, int32_t mode);
/* Constraint scan of the shared-memory kernels for n > 64 when C is not staged: 1 or -1 (default) = every CTA keeps a
 * transposed copy of its problem's C in a global-memory slice (L2-resident) and scans it with coalesced loads (measures
 * faster there), 0 = scan C in place (one strided row per thread). Same arithmetic: results are bit-identical (tests
 * cross-check both). The kernels for n <= 64 always scan in place (the transposed scan measured slower there). Also
 * selects whether the global-workspace kernel scans a transposed copy of a batch-shared C. */
int jrlqp_set_scan_transposed(jrlqp_solver * s, int32_t on);
/* Bytes of ONE instance's G that cross the host link in jrlqp_solve_batch_host (non-shared G, no factor requested):
 * the kernels read the lower triangle only, so the host entry point does not move all of G — with a pinned (page-locked,
 * mapped) caller buffer and n <= 64 the kernels read G in place (lower triangle), otherwise G is uploaded as its left
 * n/2 columns plus the bottom-right block. Environment overrides for tuning comparisons: JRLQP_G_ZEROCOPY=0|1,
 * JRLQP_H2D_FULL_G=1. */
int64_t jrlqp_host_g_bytes(const jrlqp_solver * s, int32_t pinned);
/* Number of kernels this library has launched since it was loaded (all solvers). */
int64_t jrlqp_launch_count(void);
/* Last CUDA error string seen by this solver ("" if none). */
const char * jrlqp_last_error(const jrlqp_solver * s);
int jrlqp_version(void);

/* FP64 roofline probe: runs a dependent-free DFMA loop on every SM and returns the measured
 * TFLOP/s (2 flops per FMA), or a negative error. Used by bench.py for the roofline denominator. */
double jrlqp_measure_fp64_tflops(int32_t device, int32_t repeats);

/* FP64 tensor-core experiment (jrl-qp_b200/csrc/dmma_probe.cu): a 128 x 128 x 64 product per 4-warp CTA, one CTA per SM
 * (the shape and residency of the n = 128 solver kernel), `reps` times. out6 (HOST): [0] GFLOP/s of a register-blocked
 * FP64-pipe kernel, [1] GFLOP/s of an mma.sync.m8n8k4.f64 (DMMA) kernel, [2] fraction of single-DMMA outputs equal to the
 * sequential fma chain over k, [3] ... equal to the pairwise order, [4] fraction of length-64 inner products evaluated by
 * DMMA with the canonical dot4 interleaving that equal dot4 bit for bit, [5] fraction of outputs on which the two product
 * kernels agree bit for bit. */
int jrlqp_probe_dmma(int32_t device, int32_t reps, double * out6);

/* Self-test of the short-latency exact division / square root used on the solver's serial
 * recurrences (jrl-qp_b200/csrc/fp64_exact.cuh) against the stock IEEE operations, on `samples`
 * pseudo-random operand pairs with binary exponents in [-exponent_span, exponent_span] and a
 * reciprocal perturbed by up to rcp_ulps ulps. counts5 (HOST, 5 entries): [0] quotients proven
 * correctly rounded, [1] proven yet different from x / y (must be 0), [2] unproven (the kernels
 * then use the stock division), [3] square roots different from sqrt() (must be 0), [4] reciprocal
 * square-root by-products further than 4 ulp from the true value. */
int jrlqp_selftest_arith(int32_t device, int64_t samples, uint64_t seed, int32_t exponent_span, int32_t rcp_ulps, uint64_t * counts5);

/* ------------------------------------------------------------------------------------------------
 * Warm-started SEQUENCES (SURVEY §8 f2): the reference's control-loop use case and benchmark
 * (benchmarks/SolversWarmStart.cpp:234-276): the same G, C and bounds are solved `steps` times with a
 * slowly varying linear term a(t); with warm != 0 every step after the first is warm-started from the
 * active set the previous step ended with ("as empty => reuse the previous active set",
 * src/experimental/GoldfarbIdnaniSolver.cpp:58-61), the first one from pb->as_in (nullable), through the
 * experimental solver (BENCH_GI_EX); with warm == 0 every step is a cold solve of the stable solver
 * (BENCH_GI). The whole sequence is enqueued on one stream: the active set never leaves the GPU.
 *   pb->a               linear term of step 0; step t reads pb->a + t * a_step_stride (elements)
 *   res                 outputs of the LAST step — unless a *_step_stride below is non-zero, in which
 *                       case step t writes that output at (pointer + t * stride) (elements)
 *   iterations_total    [batch] (nullable) sum of iterations() over the steps — the "it" counter of the
 *                       reference benchmark
 *   status_worst        [batch] (nullable) worst TerminationStatus over the steps
 * res->active_set is required when warm != 0 (it carries the active set from step to step).
 * G does not change along a sequence: with warm != 0 and n <= 128 the handle keeps the factor step 0 leaves (L, L^-T and
 * the diagonal: (n n + 2 n) doubles per instance, device memory owned by the handle and sized by the largest call) and
 * the later steps re-read it instead of factorising again — same operands, same bits; JRLQP_SEQ_FCACHE=0 in the
 * environment (read by jrlqp_create) turns it off. The reference refactorises on every call (its solve() overwrites G).
 * ------------------------------------------------------------------------------------------------ */
typedef struct jrlqp_sequence
{
  int32_t steps;
  int32_t warm;
  int64_t a_step_stride;
  int64_t x_step_stride; /* 0: only the last step's solution is kept */
  int64_t u_step_stride;
  int64_t f_step_stride;
  int64_t iterations_step_stride;
  int64_t status_step_stride;
  int32_t * iterations_total;
  int32_t * status_worst;
} jrlqp_sequence;
/* DEVICE pointers, asynchronous on `stream`. */
int jrlqp_solve_sequence_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res, void * stream);
/* HOST pointers: G, C, bounds and all `steps` linear terms are uploaded once, the steps run back to back
 * on the device, the requested outputs come back once. Returns the worst status over batch and steps
 * (>= 0) or a negative JRLQP_ERR_*. */
int jrlqp_solve_sequence_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res);

/* ------------------------------------------------------------------------------------------------
 * GPU-side batch verifier (SURVEY §8 f3): jrl::qp::test::testKKT (src/test/kkt.cpp:87-195:
 * stationarity |G x + a + C u_c + u_b|_inf <= tau_d (1 + |u|_inf), and per constraint one of
 * {at lower & u <= -tau_u, inside & |u| <= tau_u, at upper & u >= tau_u} with tau_x = tau_p (1 + |x|_inf))
 * and the planted-solution comparison of the reference's tests (x.isApprox(x_ref, prec),
 * tests/GoldfarbIdnaniSolverTest.cpp:94-97), for a batch resident in HBM. Uses the FULL matrix G
 * (both triangles), as the reference does.
 *   flags  [batch]     bit 0: stationarity holds, bit 1: feasibility / complementarity holds,
 *                      bit 2: x ~ x_ref (only when x_ref is given)
 *   resid  [batch][4]  (nullable) |dL|_inf, tau_u, tau_x, |x - x_ref|^2
 *   n_fail             (nullable) number of instances with a missing bit. _device: a DEVICE counter the
 *                      caller has zeroed; _host: a host int64.
 * ------------------------------------------------------------------------------------------------ */
typedef struct jrlqp_kkt_args
{
  int32_t n, mc, use_bounds;
  double tau_p, tau_d; /* 1e-6, 1e-6 (include/jrl-qp/test/kkt.h:83-84) */
  double prec; /* 1e-6 */
  const double * x; /* [batch][n] */
  const double * u; /* [batch][mc+nb], reference sign convention (DualSolver::multipliers) */
  const double * x_ref; /* [batch][n], nullable */
  int32_t * flags;
  double * resid;
  int64_t * n_fail;
} jrlqp_kkt_args;
void jrlqp_kkt_default_args(jrlqp_kkt_args * k);
int jrlqp_kkt_check_device(const jrlqp_problem * pb, const jrlqp_kkt_args * k, int32_t device, void * stream);
/* Host pointers (uploads the batch; a verifier, not a hot path). Returns the number of failing
 * instances (>= 0, saturating) or a negative JRLQP_ERR_*. */
int jrlqp_kkt_check_host(const jrlqp_problem * pb, const jrlqp_kkt_args * k, int32_t device);

/* ------------------------------------------------------------------------------------------------
 * Structured Cholesky decompositions (north-star item 4), batched: `batch` matrices that share ONE
 * block structure are factorised / solved by one call, one instance per CTA.
 *
 * Replaces structured::StructuredG (include/jrl-qp/structured/StructuredG.h:14-76,
 * src/structured/StructuredG.cpp:6-113) and the functions it dispatches to:
 *   decomposition::triBlockDiagLLT / triBlockDiagLSolve / triBlockDiagLTransposeSolve
 *       (include/jrl-qp/decomposition/triBlockDiagLLT.h:41-72, src/decomposition/triBlockDiagLLT.cpp)
 *   decomposition::blockArrowLLT / blockArrowLSolve / blockArrowLTransposeSolve
 *       (include/jrl-qp/decomposition/blockArrowLLT.h:72-110, src/decomposition/blockArrowLLT.cpp)
 * The reference passes std::vector<MatrixRef> views; the descriptor below carries the same views
 * as (element offset from the instance base, leading dimension) per block, so blocks may be views
 * into a dense matrix (tests/triBlockDiagLLTTest.cpp:41-43) or packed tiles.
 * ------------------------------------------------------------------------------------------------ */

/* structured::StructuredG::Type (include/jrl-qp/structured/StructuredG.h:17-22), same order */
enum jrlqp_structure_type
{
  JRLQP_TRI_BLOCK_DIAGONAL = 0,
  JRLQP_BLOCK_ARROW_UP = 1,
  JRLQP_BLOCK_ARROW_DOWN = 2
};

/* HOST arrays (copied at create). Diagonal block i is block_size[i] x block_size[i] (lower triangle
 * read and written; the upper part "remains whatever was there", triBlockDiagLLT.h:37-39).
 * Off-diagonal block i (i < nblocks-1), column-major with leading dimension off_ld[i]:
 *   TRI_BLOCK_DIAGONAL  S_i  n_{i+1} x n_i   sub-diagonal block (i+1, i)
 *   BLOCK_ARROW_DOWN    S_i  n_{b-1} x n_i   block of the last block row
 *   BLOCK_ARROW_UP      S_i  n_{i+1} x n_0   block of the first block column (holds B_i^T afterwards)
 */
typedef struct jrlqp_structure
{
  int32_t type; /* jrlqp_structure_type */
  int32_t nblocks;
  const int32_t * block_size; /* [nblocks]   */
  const int64_t * diag_offset; /* [nblocks]   elements from the instance base */
  const int32_t * diag_ld; /* [nblocks]   */
  const int64_t * off_offset; /* [nblocks-1] */
  const int32_t * off_ld; /* [nblocks-1] */
} jrlqp_structure;

typedef struct jrlqp_structured jrlqp_structured;

/* StructuredG(Type, diag, offDiag) (src/structured/StructuredG.cpp:6-20). batch_capacity bounds
 * the *_host entry points (device staging is allocated on first use). Blocks up to 96 rows
 * (three tiles of the largest block must fit in the 227 KB of shared memory of one SM). */
int jrlqp_structured_create(jrlqp_structured ** out, const jrlqp_structure * st, int64_t batch_capacity, int32_t device);
int jrlqp_structured_destroy(jrlqp_structured * s);
const char * jrlqp_structured_last_error(const jrlqp_structured * s);

/* StructuredG::lltInPlace (src/structured/StructuredG.cpp:22-43), in place on `data`
 * (instance k at data + k * stride). ok[k] (nullable) = 1 if decomposed, 0 if a diagonal block was
 * not positive definite (the reference returns false; the failing block and the ones after it are
 * then unspecified). DEVICE pointers, asynchronous on `stream`. */
int jrlqp_structured_llt_device(jrlqp_structured * s, double * data, int64_t stride, int64_t batch, int32_t * ok, void * stream);
/* Same with HOST pointers (H2D, kernel, D2H, synchronise). Returns the number of instances that
 * failed (>= 0) or a negative JRLQP_ERR_*. */
int jrlqp_structured_llt_host(jrlqp_structured * s, double * data, int64_t stride, int64_t batch, int32_t * ok);

/* StructuredG::solveL (transpose = 0: X = (P L)^-1 M, src/structured/StructuredG.cpp:66-113) and
 * StructuredG::solveInPlaceLTranspose (transpose = 1: X = P L^-T M, :45-64), in place on M
 * (n x ncols column-major, leading dimension ldm, instance k at M + k * m_stride). start / end are
 * the reference's hints: rows [start, end) of M are the only non-zero ones (end < 0: none given);
 * they only skip work, results are those of the plain call. `data` holds the factor. */
int jrlqp_structured_solve_device(jrlqp_structured * s,
                                  const double * data,
                                  int64_t stride,
                                  double * M,
                                  int32_t ldm,
                                  int32_t ncols,
                                  int64_t m_stride,
                                  int64_t batch,
                                  int32_t transpose,
                                  int32_t start,
                                  int32_t end,
                                  void * stream);
int jrlqp_structured_solve_host(jrlqp_structured * s,
                                const double * data,
                                int64_t stride,
                                double * M,
                                int32_t ldm,
                                int32_t ncols,
                                int64_t m_stride,
                                int64_t batch,
                                int32_t transpose,
                                int32_t start,
                                int32_t end);
/* threads per instance, resident instances per SM and shared memory per instance of the two kernels */
typedef struct jrlqp_structured_info
{
  int32_t threads;
  int32_t llt_smem_bytes, llt_ctas_per_sm;
  int32_t solve_smem_bytes, solve_ctas_per_sm;
  int32_t num_sms;
  int64_t elements_per_instance; /* doubles of the factor actually touched (algorithmic bytes / 8) */
} jrlqp_structured_info;
/* Kernel used by jrlqp_structured_llt_*: 0 automatic, 1 the general kernel (one CTA per instance, tiles in shared memory),
 * 2 the small-tile kernel (tri-block-diagonal chains of uniform dense 8 / 12 / 16-row tiles: two instances per warp, tiles in
 * registers), 3 the same with the tiles of the next block fetched by TMA bulk copies (cp.async.bulk + mbarrier). All
 * produce the same bits. Environment override at creation: JRLQP_STRUCT_KERNEL. */
int jrlqp_structured_set_kernel(jrlqp_structured * s, int32_t mode);
int jrlqp_structured_get_info(const jrlqp_structured * s, jrlqp_structured_info * info);

/* ---------------------------------------------------------------------------------------------
 * Structured solver: experimental::BlockGISolver, batched.
 *
 * Replaces experimental::BlockGISolver::solve(StructuredG, a, StructuredC, bl, bu, xl, xu, as)
 * (include/jrl-qp/experimental/BlockGISolver.h:24-46, src/experimental/BlockGISolver.cpp:18-60) and what it
 * runs on: structured::StructuredJ (src/structured/StructuredJ.cpp:33-57), structured::StructuredQR
 * (src/structured/StructuredQR.cpp:66-103), structured::StructuredC (src/structured/StructuredC.cpp:9-77),
 * internal::OrthonormalSequence (src/internal/OrthonormalSequence.cpp:50-196) and the DualSolver loop
 * (src/DualSolver.cpp:91-168): the dual active-set method with J = L^-T Q kept implicit — L the structured
 * factor of G, Q a sequence of Householder reflectors (activations) and Givens sequences (drops).
 * As in the reference, the solver handles cold starts of problems WITHOUT equalities: the reference asserts
 * that no constraint is active after the initial scan (BlockGISolver.cpp:474); an instance whose data contain
 * bl == bu or xl == xu is reported as JRLQP_INCONSISTENT_INPUT. Instances that exhaust the storage of the
 * orthonormal sequence (2 n max_iter doubles per resident CTA) report JRLQP_UNKNOWN.
 * Sizes: n <= 1024 variables, diagonal blocks of 1 ... 96 rows; jrlqp_blockgi_create returns JRLQP_ERR_ARG for a
 * larger n, and for a problem whose per-CTA state (which grows with n, the largest block and max_iter) does not fit
 * in the shared memory of one CTA.
 * --------------------------------------------------------------------------------------------- */

/* structured::StructuredC(std::vector<MatrixConstRef>) (src/structured/StructuredC.cpp:9-25): block-diagonal
 * constraint matrix. Block i is nvar[i] x ncstr[i], column-major (one constraint normal per column), at
 * `offset[i]` elements from the instance base, leading dimension ld[i]. HOST arrays, copied at create. The
 * nvar[i] must add up to the size of G; constraints are numbered block after block. */
typedef struct jrlqp_cstructure
{
  int32_t nblocks;
  const int32_t * nvar;
  const int32_t * ncstr;
  const int64_t * offset;
  const int32_t * ld;
} jrlqp_cstructure;

/* One batch of structured problems; strides in ELEMENTS between instances, 0 = shared.
 *   G  the blocks described by the jrlqp_structure given at create. With G_stride != 0 the blocks are
 *      factorised IN PLACE, as the reference's pb_.G.lltInPlace() does on the caller's views
 *      (BlockGISolver.cpp:71); a shared G (stride 0) is left untouched (one private copy is factorised).
 *      The *_host entry point never writes to the caller's G.
 *   C  the blocks described by the jrlqp_cstructure. */
typedef struct jrlqp_block_problem
{
  int64_t batch;
  double * G;
  int64_t G_stride;
  const double * a;
  int64_t a_stride;
  const double * C;
  int64_t C_stride;
  const double * bl;
  int64_t bl_stride;
  const double * bu;
  int64_t bu_stride;
  const double * xl; /* NULL <=> created without bounds */
  int64_t xl_stride;
  const double * xu;
  int64_t xu_stride;
} jrlqp_block_problem;

typedef struct jrlqp_blockgi jrlqp_blockgi;

/* BlockGISolver(nbVar, nbCstr, useBounds) (src/experimental/BlockGISolver.cpp:12-15) for one block structure. */
int jrlqp_blockgi_create(jrlqp_blockgi ** out, const jrlqp_structure * G, const jrlqp_cstructure * C, int32_t use_bounds,
                         int64_t batch_capacity, int32_t device);
int jrlqp_blockgi_destroy(jrlqp_blockgi * s);
const char * jrlqp_blockgi_last_error(const jrlqp_blockgi * s);
/* DualSolver::options (max_iter, big_bnd; warm_start must be 0: see above) */
int jrlqp_blockgi_set_options(jrlqp_blockgi * s, const jrlqp_options * opt);
int jrlqp_blockgi_get_options(const jrlqp_blockgi * s, jrlqp_options * opt);
/* solve() + the DualSolver accessors for the batch; jrlqp_result as for the dense solver (result.L is ignored:
 * the factor is left in G). DEVICE pointers, asynchronous on `stream`. */
int jrlqp_blockgi_solve_device(jrlqp_blockgi * s, const jrlqp_block_problem * pb, const jrlqp_result * res, void * stream);
/* Same with HOST pointers; returns the worst jrlqp_termination_status (>= 0) or a negative JRLQP_ERR_*. */
int jrlqp_blockgi_solve_host(jrlqp_blockgi * s, const jrlqp_block_problem * pb, const jrlqp_result * res);

typedef struct jrlqp_blockgi_info
{
  int32_t n, mc, nb;
  int32_t threads; /* per QP (one QP per CTA) */
  int32_t smem_bytes, ctas_per_sm, grid, num_sms;
  int64_t workspace_bytes_per_cta; /* packed R + storage of the orthonormal sequence */
  int64_t g_elements_per_instance;
} jrlqp_blockgi_info;
int jrlqp_blockgi_get_info(const jrlqp_blockgi * s, jrlqp_blockgi_info * info);

/* Test harness of internal::OrthonormalSequence as the structured solver stores it (tests/InternalTest.cpp:35-323): the
 * kernel's own applyToTheLeft (transpose = 0) / applyTransposeToTheLeft (1) on `ncases` HOST vectors v [ncases][n], in
 * place. rec: nrec triples (start, size, offset into qdata); Householder record: start >= 0, `size` entries
 * [tau, essential(size-1)] — H = I - tau e e^T, e = [1; essential] embedded at `start`; Givens record: start | 0x80000000,
 * `size` rotations on the rows (start + i, start + i + 1), data [c(size), s(size)]. */
int jrlqp_blockgi_test_sequence(int32_t device, int32_t n, int32_t nrec, const int32_t * rec, const double * qdata, int64_t qlen, double * v,
                                int32_t ncases, int32_t transpose, int32_t threads);

/* ---------------------------------------------------------------------------------------------------------------
 * Multi-GPU: one handle, one HOST batch, every GPU of the box (SURVEY.md §8e: "contiguous batch ranges per GPU, one
 * host thread or stream set per device, host-side scatter/gather; no collective"). The reference solves one QP per
 * call on one thread (src/GoldfarbIdnaniSolver.cpp:18-54); a caller that loops over a batch of them — the pattern of
 * benchmarks/Solvers.cpp:513-518 — hands the whole batch to jrlqp_multi_solve_batch_host instead:
 *   scatter  shard k = instances [lo_k, hi_k) (sizes differ by at most one; jrlqp_multi_shard returns the range) is a
 *            VIEW of the caller's arrays (pointer + lo_k * stride; arrays shared by the batch, stride 0, go to every
 *            device once), solved on device k by its own jrlqp_solver — own streams, own device staging — driven by a
 *            persistent host thread per device;
 *   gather   every device writes its results straight into the caller's arrays at [lo_k, hi_k): no extra copy.
 * devices == NULL: devices 0 .. n_devices-1 (n_devices <= 0: all visible). batch_capacity bounds the batch of a call.
 * Same semantics, statuses and bits as jrlqp_solve_batch_host on one device (tests/test_gpu_multi.py). */
typedef struct jrlqp_multi jrlqp_multi;
int jrlqp_multi_create(jrlqp_multi ** out, int32_t n, int32_t mc, int32_t use_bounds, int64_t batch_capacity, const int32_t * devices,
                       int32_t n_devices);
int jrlqp_multi_destroy(jrlqp_multi * m);
int jrlqp_multi_set_options(jrlqp_multi * m, const jrlqp_options * opt);
int jrlqp_multi_device_count(const jrlqp_multi * m);
int jrlqp_multi_device(const jrlqp_multi * m, int32_t k); /* CUDA ordinal of shard k */
jrlqp_solver * jrlqp_multi_solver(jrlqp_multi * m, int32_t k); /* the per-device solver (introspection, tuning switches) */
/* The range [begin, end) of a batch of `batch` instances that shard k receives in the NEXT call. */
int jrlqp_multi_shard(const jrlqp_multi * m, int64_t batch, int32_t k, int64_t * begin, int64_t * end);
/* Load balancing (default on): the shares of the shards start equal (sizes differ by at most one) and then follow the
 * throughput every device achieved in the previous calls of this handle — the GPUs of one box need not see the same
 * host-link bandwidth (profiles/r02n_multi_e2e.txt). A share never exceeds 1.5 / n_devices. Results do not depend on
 * the sharding. on = 0 restores equal shards. jrlqp_multi_get_weights: the current shares (n_devices doubles, sum 1). */
int jrlqp_multi_set_balancing(jrlqp_multi * m, int32_t on);
int jrlqp_multi_get_weights(const jrlqp_multi * m, double * weights);
/* Returns the worst jrlqp_termination_status over the whole batch (>= 0) or a negative JRLQP_ERR_*. */
int jrlqp_multi_solve_batch_host(jrlqp_multi * m, const jrlqp_problem * pb, const jrlqp_result * res);
int jrlqp_multi_solve_batch_warm_host(jrlqp_multi * m, const jrlqp_problem * pb, const jrlqp_result * res);
const char * jrlqp_multi_last_error(const jrlqp_multi * m);

/* Platform probe behind the end-to-end numbers: aggregate GB/s of concurrent pinned-host <-> device copies over
 * n_devices GPUs (devices == NULL: 0 .. n_devices-1), `bytes` per device and repetition, `reps` repetitions back to
 * back on one stream per device. direction: 0 host -> device, 1 device -> host, 2 both at once (sum of the two).
 * per_device (nullable, n_devices entries) receives every device's own GB/s. Negative on error. */
double jrlqp_measure_host_link(const int32_t * devices, int32_t n_devices, int64_t bytes, int32_t reps, int32_t direction, double * per_device);

#ifdef __cplusplus
}
#endif

#endif /* JRLQP_B200_H */
