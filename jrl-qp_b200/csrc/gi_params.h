// Kernel parameter block shared by the host API (capi.cu) and the device code.
#pragma once
#include <stdint.h>

namespace jrlqp
{

// jrl::qp::ActivationStatus / TerminationStatus values (include/jrl-qp/enums.h:14-37)
enum : int
{
  ST_INACTIVE = 0,
  ST_LOWER = 1,
  ST_UPPER = 2,
  ST_EQUALITY = 3,
  ST_LOWER_BOUND = 4,
  ST_UPPER_BOUND = 5,
  ST_FIXED = 6
};
enum : int
{
  TS_SUCCESS = 0,
  TS_INCONSISTENT_INPUT = 1,
  TS_NON_POS_HESSIAN = 2,
  TS_INFEASIBLE = 3,
  TS_MAX_ITER_REACHED = 4,
  TS_LINEAR_DEPENDENCY_DETECTED = 5,
  TS_OVERCONSTRAINED_PROBLEM = 6,
  TS_UNKNOWN = 7
};

// Shared-memory layout of the dense kernels (gi_dense_cta.cuh), computed on the host (capi.cu: make_layout); in doubles
// unless noted. The offset of each field within the parameter block decides how the compiler pairs the kernels' 64- and
// 128-bit loads of them: `pad` and the place of total_doubles keep those offsets, and so the kernels' machine code.
struct DenseSmem
{
  int ldj; // leading dimension of the row-major J/L buffer (odd => conflict-free row-strided access)
  int ldcs; // leading dimension of the staged C (odd), if staged
  int npad; // threads per CTA (>= n)
  int off_R, off_x, off_z, off_d, off_r, off_u, off_cv;
  int pad[2];
  int off_gcs, off_ldiag, off_rinv, off_scr, off_C, off_alist;
  int total_doubles; // (host only)
  int off_iscr, off_stat, off_eq, off_il; // int / int8 / uint16 arrays
  int off_V, off_bact, off_hco, off_alpha; // warm-start kernels only
};

struct GiParams
{
  // sizes
  int n, mc, nb;
  int ldg, ldc;
  long long batch;
  // options
  int max_iter;
  double big_bnd;
  // inputs (device pointers, element strides between instances; 0 = shared)
  const double * G;
  long long sG;
  const double * a;
  long long sa;
  const double * C;
  long long sC;
  const double * bl;
  long long sbl;
  const double * bu;
  long long sbu;
  const double * xl;
  long long sxl;
  const double * xu;
  long long sxu;
  const signed char * as_in; // warm start: initial activation status guess (nullable), int8 x (mc + nb)
  long long s_as;
  int warm_start; // SolverOptions::warmStart_
  // outputs (device pointers, dense; nullable except x)
  double * x;
  double * u;
  double * f;
  int * iterations;
  int * status;
  signed char * active_set;
  int * active_list;
  int * n_active;
  double * L;
  // global-memory workspace of the large-n kernel (gi_large.cuh): one slice of work_stride doubles per CTA
  double * work;
  long long work_stride;
  int * work_busy; // one flag per slice: a CTA claims a free slice when it starts and releases it when it exits
  int work_slots;
  int ring_cols; // large-n kernel: columns of J per stage of the TMA-fed column ring (gi_large.cuh: ring_*), 0 = off
  int slab_rows; // large-n WARM kernel: rows of J per shared-memory slab of J = J Q (gi_large_warm.inl: warm_JQ_slab), 8 / 16, 0 = off
  // factor of a batch-shared G (sG == 0), large-n kernel: computed once by gi_large_prefactor_kernel, copied by the CTAs.
  // Layout (doubles, ldl = n rounded up to 4): [0, n ldl) J = L^-T column-major (upper triangle, rest 0),
  // [n ldl, 2 n ldl) scratch of the prefactor kernel, [2 n ldl, 3 n ldl) L column-major, then diag(L) [nv], 1 / diag(L) [nv]
  const double * pre;
  const int * pre_ok; // 1: G is positive definite
  // transposed copy of C for the coalesced constraint scan (gi_dense_cta.cuh, non-staged kernels): one slice of
  // ct_stride doubles per resident CTA (groups of 128 constraints, layout: ct_offset in gi_dense_cta.cuh), claimed like the
  // work slices; null = scan C in place. Large-n kernel: one copy of a batch-shared C for the whole launch (ct_slots == 0)
  double * ct;
  long long ct_stride;
  int * ct_busy;
  int ct_slots;
  int ldct;
  // warm-started sequences (jrlqp_solve_sequence_*): G does not change from step to step, so the factor of step 0 — L below the
  // diagonal, J = L^-T above it, diag(L) and its reciprocals: n n + 2 n doubles per instance — is kept in HBM and re-read by the
  // later steps instead of being recomputed (fcache_mode 0: off, 1: compute and store, 2: load). diag(L)[0] = -1 marks an
  // instance whose G is not positive definite.
  double * fcache;
  long long fcache_stride;
  int fcache_mode;
  // persistent work queue
  unsigned long long * counter;
  unsigned long long * phase_cycles; // [4 warps][16 phases], only with -DJRLQP_PHASE_TIMING (else null)
  DenseSmem lay; // dense kernels only
};

} // namespace jrlqp
