// Host side of the C-ABI (include/jrlqp_b200.h): solver handle, shared-memory layout, kernel
// dispatch, and the host-pointer entry point that pipelines H2D copies, the persistent kernel and
// D2H copies over a few streams. Pure CUDA runtime — no PyTorch, no CPU fallback.
#include "smem_limit.hpp"
#include "gi_dense_cta.cuh"
#include "gi_large.cuh"
#include "jrlqp_b200.h"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace jrlqp;

namespace
{

static int g_seq_fcache = 1; // JRLQP_SEQ_FCACHE=0: every step of a warm-started sequence factorises again (A/B, tests)
static int g_zero_copy_G = -1; // kernels read G from the caller's pinned host buffer: 1 on, 0 off, -1 automatic (n <= 64); JRLQP_G_ZEROCOPY
static bool g_h2d_lower = true; // host entry points upload only what the kernels read of G (see h2d_G)
std::atomic<long long> g_launches{0};

constexpr int kStreams = 3;
constexpr int kMaxChunks = 64;

using KernelFn = void (*)(const GiParams);

KernelFn pick_warm_kernel(int warps)
{
  switch(warps)
  {
    case 1:
      return gi_dense_cta_kernel<1, false, true>;
    case 2:
      return gi_dense_cta_kernel<2, false, true>;
    case 3:
      return gi_dense_cta_kernel<3, false, true>;
    case 4:
      return gi_dense_cta_kernel<4, false, true>;
    default:
      return nullptr;
  }
}

KernelFn pick_kernel(int warps, bool stage)
{
  switch(warps)
  {
    case 1:
      return stage ? gi_dense_cta_kernel<1, true> : gi_dense_cta_kernel<1, false>;
    case 2:
      return stage ? gi_dense_cta_kernel<2, true> : gi_dense_cta_kernel<2, false>;
    case 3:
      return stage ? gi_dense_cta_kernel<3, true> : gi_dense_cta_kernel<3, false>;
    case 4:
      return stage ? gi_dense_cta_kernel<4, true> : gi_dense_cta_kernel<4, false>;
    default:
      return nullptr;
  }
}

DenseSmem make_layout(int n, int mc, int nb, int warps, bool stage, bool warm = false)
{
  DenseSmem L{};
  L.ldj = n | 1;
  L.ldcs = n | 1;
  L.npad = 32 * warps;
  const int np = L.npad;
  int o = n * L.ldj;
  L.off_R = o;
  o += n * (n + 1) / 2;
  o += o & 1; // the vectors start 16-byte aligned (128-bit loads of broadcast operands)
  L.off_x = o;
  o += np;
  L.off_z = o;
  o += np;
  L.off_d = o;
  o += np;
  L.off_r = o;
  o += np;
  L.off_u = o;
  o += np + 2;
  L.off_cv = o;
  o += np;
  o += o & 1; // 16-byte alignment of the per-link records of the Givens sweep
  L.off_gcs = o; // (one array of 32-byte records: see GiCta::givens_recurrence)
  o += 4 * np;
  L.off_ldiag = o;
  o += np;
  L.off_rinv = o;
  o += np;
  L.off_scr = o;
  o += 16;
  L.off_C = o;
  o += stage ? mc * L.ldcs : 0;
  L.off_alist = o;
  o += np / 2 + 1;
  L.off_iscr = o;
  o += 8;
  L.off_stat = o;
  o += (mc + nb + 7) / 8 + 1;
  L.off_eq = o;
  o += (mc + nb + 7) / 8 + 1;
  L.off_il = o; // uint16 per general constraint
  o += (mc + 3) / 4;
  L.off_V = L.off_bact = L.off_hco = L.off_alpha = o;
  if(warm)
  {
    L.off_V = o;
    o += n * (n - 1) / 2 + 1;
    L.off_bact = o;
    o += np;
    L.off_hco = o;
    o += np;
    L.off_alpha = o;
    o += np;
  }
  L.total_doubles = o;
  return L;
}

// Everything a launch of one kind of call (cold or warm) needs: the kernel, its size and residency, and either the
// shared-memory layout of the dense kernel or the per-CTA workspace of the global-workspace (large-n) kernel.
struct LaunchCfg
{
  KernelFn fn = nullptr; // null: not configured
  int threads = 0, smem = 0, occ = 0, regs = 0; // per CTA: threads, dynamic shared-memory bytes; resident CTAs per SM; registers
  bool large = false; // the global-workspace kernel (gi_large.cuh)
  // dense kernel
  bool stage = false; // C staged in shared memory
  DenseSmem lay{};
  // large-n kernel
  int ring_cols = 0; // columns per stage of the TMA column ring (0: off)
  int slab_rows = 0; // rows per slab of J = J Q, warm kernel (0: off)
  double * work = nullptr;
  int * busy = nullptr;
  int work_slots = 0;
  long long work_stride = 0;
};

// What a call asks of launch() besides its problem and result
struct CallArgs
{
  bool warm = false; // the warm-start capable solver
  bool force_warm_start = false; // honour as_in whatever options().warm_start says (sequences)
  bool pre_ready = false; // the factor of a shared G and the transposed shared C were prepared earlier on the stream
  int fcache_mode = 0; // sequence factor cache (gi_params.h: fcache_mode)
};

} // namespace

namespace jrlqp
{
void count_launch()
{
  g_launches.fetch_add(1);
}
} // namespace jrlqp

struct jrlqp_solver
{
  int n = 0, mc = 0, nb = 0, m = 0;
  long long capacity = 0;
  int device = 0;
  jrlqp_options opt{};
  int warps = 1;
  int stage_mode = -1; // -1 auto
  int path_mode = 0; // 0 automatic (n <= 128: shared-memory kernel), 1 shared-memory kernel, 2 global-workspace kernel
  // [cold, warm]: what serves each kind of call. Cold: configured at creation and by set_kernel_path / set_stage_c. Warm
  // (experimental solver): configured on the first warm call, reset by set_kernel_path.
  LaunchCfg cfg[2];
  // [cold, warm]: the global-workspace kernel of each family, configured on first use; its workspace lives as long as the handle
  LaunchCfg large_cfg[2];
  signed char * d_as = nullptr; // staging of as_in for the host entry point
  // warm-started sequences (jrlqp_solve_sequence_*): scratch for per-step iterations / status and host staging
  double * d_fcache = nullptr; // factor of step 0 of a warm-started sequence (gi_params.h: fcache), re-read by the later steps
  long long fcache_cap = 0; // doubles
  int * d_seq_it = nullptr;
  int * d_seq_status = nullptr;
  long long cap_seq = 0;
  double * d_seq = nullptr; // arena: linear terms of all steps + per-step outputs (host entry point)
  long long cap_seq_arena = 0;
  int * d_seq_tot = nullptr; // [2][capacity]: iterations_total, status_worst (host entry point)
  double * d_cts = nullptr; // transposed copy of a batch-shared C (large-n kernel)
  int ldcts = 0;
  double * d_pre = nullptr; // factor of a batch-shared G (large-n kernel), see gi_params.h
  int * d_pre_ok = nullptr;
  int pre_smem = 0;
  // capacity (instances) of every staging buffer of the host entry point: 1 for arrays shared by the batch
  long long cap_G = 0, cap_a = 0, cap_C = 0, cap_bl = 0, cap_bu = 0, cap_xl = 0, cap_xu = 0, cap_out = 0, cap_L = 0;
  // transposed copy of C for the coalesced constraint scan of the non-staged shared-memory kernels
  int scan_transposed = -1; // 1: scan the CTA's transposed copy of C, 0: scan C in place, -1: automatic (transposed for n > 64)
  double * d_ct = nullptr;
  int * d_ct_busy = nullptr;
  int ct_slots = 0, ldct = 0;
  long long ct_stride = 0;
  int num_sms = 0;
  int max_smem_optin = 0;
  // device-side scratch
  unsigned long long * d_counters = nullptr; // kMaxChunks counters
  unsigned long long * d_phase = nullptr; // per-phase cycle counters (debug builds with -DJRLQP_PHASE_TIMING)
  int next_counter = 0;
  // staging for the host entry point
  double *d_G = nullptr, *d_a = nullptr, *d_C = nullptr, *d_bl = nullptr, *d_bu = nullptr, *d_xl = nullptr, *d_xu = nullptr;
  double *d_x = nullptr, *d_u = nullptr, *d_f = nullptr, *d_L = nullptr;
  int *d_it = nullptr, *d_status = nullptr, *d_alist = nullptr, *d_nact = nullptr;
  signed char * d_act = nullptr;
  bool staging_ready = false;
  cudaStream_t streams[kStreams] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_shared = nullptr;
  // device entry points: calls on ONE handle are serialised on the device (per-handle scratch — prefactor of a shared G,
  // transposed shared C, sequence counters — is single-buffered): a call on a different stream first waits for the last one
  cudaEvent_t ev_last = nullptr;
  cudaStream_t last_stream = nullptr;
  bool has_last = false;
  std::string err;

  bool check(cudaError_t e, const char * what)
  {
    if(e == cudaSuccess) return true;
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
  }
};

#define CK(call)                             \
  do                                         \
  {                                          \
    if(!s->check((call), #call)) return JRLQP_ERR_CUDA; \
  } while(0)

static constexpr int kLargeThreads = 256;

// CTAs of `fn` resident per SM at `threads` threads and `smem` bytes of dynamic shared memory; 0 when that size does not
// fit (the error of the failed call cleared).
static int resident_ctas(const jrlqp_solver * s, KernelFn fn, int threads, int smem)
{
  int occ = 0;
  if(smem > s->max_smem_optin) return 0;
  if(jrlqp::raise_smem_limit(fn, smem) != cudaSuccess || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, threads, smem) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return occ;
}

// Large-n kernel: shared-memory size, residency and the per-CTA global workspace
static int configure_large(jrlqp_solver * s, bool warm, LaunchCfg & c)
{
  KernelFn fn = warm ? gi_large_kernel<kLargeThreads, true> : gi_large_kernel<kLargeThreads, false>;
  const LargeSmem lay(s->n, s->m, warm);
  const int smem = lay.total * 8;
  if(smem > s->max_smem_optin)
  {
    s->err = "large-n kernel: the vectors do not fit in shared memory";
    return JRLQP_ERR_ARG;
  }
  int occ = resident_ctas(s, fn, kLargeThreads, smem);
  if(occ < 1)
  {
    s->err = "large-n kernel cannot be made resident";
    return JRLQP_ERR_ARG;
  }
  const int slots = occ * s->num_sms; // every resident CTA of this kernel, whatever the launch, finds a slice
  occ = std::min(occ, 2);
  // The streaming passes over J (rotation sweep of an add, z = J2 d2) read their columns through a ring of shared-memory stages
  // filled by TMA bulk copies (gi_large.cuh: ring_*), when the rows fit two per thread and the stages cost no residency.
  int smem_total = smem;
  c.ring_cols = 0;
  {
    // Measured (profiles/r5i_*, 32 768 QPs): n = 387 cold 109.4 k -> 132.1 k QP/s (+21 %: 296 workspaces of 1.2 MB do not fit L2, the
    // sweeps wait on HBM); n = 210 cold -3 % (104 MB of workspaces stay in L2 and the stages take 40 KB of L1 away), warm starts
    // of the MultiIK fixtures (zero iterations: no sweep at all) -3.5 % / 0 %. Automatic: cold kernel, n >= 256.
    // JRLQP_LARGE_RING=0: never, =2: whenever it fits.
    const char * e = getenv("JRLQP_LARGE_RING");
    const bool want = e ? (e[0] == '2' || (e[0] != '0' && !warm && s->n >= 256)) : (!warm && s->n >= 256);
    const long long ldl = (s->n + 3) & ~3ll;
    int rc = (int)std::min<long long>(16, (16384 / (ldl * 8))) & ~3;
    if(want && s->n <= 2 * kLargeThreads && rc >= 4)
    {
      const int with_ring = ((lay.total + 1) & ~1) * 8 + (int)jrlqp::large_ring_doubles(s->n, rc) * 8;
      if(resident_ctas(s, fn, kLargeThreads, with_ring) >= occ)
      {
        c.ring_cols = rc;
        smem_total = with_ring;
      }
    }
  }
  c.slab_rows = 0;
  if(warm)
  {
    // J = J Q of the warm start on slabs of 16 / 8 rows of J in shared memory (gi_large_warm.inl: warm_JQ_slab), when they cost
    // no residency. JRLQP_LARGE_SLAB=0: off (the thread = row version on the global workspace).
    const char * e = getenv("JRLQP_LARGE_SLAB");
    if(!e || e[0] != '0')
    {
      const int base = smem_total == smem ? ((lay.total + 1) & ~1) * 8 : smem_total;
      for(int R : {16, 8})
      {
        const long long bytes = jrlqp::large_slab_doubles(s->n, R) * 8;
        if(bytes > 36 * 1024) continue;
        const int tot = base + (int)bytes;
        if(resident_ctas(s, fn, kLargeThreads, tot) >= occ)
        {
          c.slab_rows = R;
          smem_total = tot;
          break;
        }
      }
    }
  }
  cudaFuncAttributes attr;
  CK(cudaFuncGetAttributes(&attr, fn));
  c.regs = attr.numRegs;
  c.threads = kLargeThreads;
  c.smem = smem_total;
  c.occ = occ;
  c.large = true;
  c.work_stride = large_workspace_doubles(s->n, warm);
  c.work_slots = slots;
  CK(cudaMalloc(&c.busy, sizeof(int) * (size_t)slots));
  CK(cudaMemset(c.busy, 0, sizeof(int) * (size_t)slots));
  CK(cudaMalloc(&c.work, sizeof(double) * (size_t)c.work_stride * (size_t)slots));
  c.fn = fn;
  return JRLQP_OK;
}

// Calls of one family (cold / warm) take the large-n kernel: configured, and its workspace allocated, on first use
static int use_large(jrlqp_solver * s, bool warm)
{
  LaunchCfg & c = s->large_cfg[warm];
  if(!c.fn)
  {
    int rc = configure_large(s, warm, c);
    if(rc != JRLQP_OK) return rc;
  }
  s->cfg[warm] = c;
  return JRLQP_OK;
}

// Cold calls
static int configure_kernel(jrlqp_solver * s)
{
  if(s->n > 128 && s->path_mode == 1)
  {
    s->err = "the shared-memory kernel needs n <= 128";
    return JRLQP_ERR_ARG;
  }
  if(s->path_mode == 2 || (s->path_mode == 0 && s->n > 128)) return use_large(s, false);
  // choose staging of C: automatic mode stages it when that costs no residency
  const int threads = 32 * s->warps;
  const DenseSmem layN = make_layout(s->n, s->mc, s->nb, s->warps, false), layS = make_layout(s->n, s->mc, s->nb, s->warps, true);
  const int smN = layN.total_doubles * 8, smS = layS.total_doubles * 8;
  const int occN = resident_ctas(s, pick_kernel(s->warps, false), threads, smN);
  const int occS = s->mc > 0 ? resident_ctas(s, pick_kernel(s->warps, true), threads, smS) : 0;
  bool stage;
  if(s->stage_mode == 0)
    stage = false;
  else if(s->stage_mode == 1)
    stage = occS > 0;
  else
    stage = occS > 0 && occS >= occN; // automatic: stage only when residency is not reduced
  KernelFn fn = pick_kernel(s->warps, stage);
  int occ = stage ? occS : occN;
  if(s->warps == 3 && occ > 0)
  {
    // register-capped instantiation of the three-warp kernel: taken when it makes more QPs resident (with C staged only
    // if that costs no residency, as above)
    const int ocN = resident_ctas(s, gi_dense_cta_kernel<3, false, false, 4>, threads, smN);
    const int ocS = (s->stage_mode != 0 && occS > 0) ? resident_ctas(s, gi_dense_cta_kernel<3, true, false, 4>, threads, smS) : 0;
    const bool cstage = s->stage_mode == 1 ? ocS > 0 : (ocS > 0 && ocS >= ocN);
    const int occC = cstage ? ocS : ocN;
    if(occC > occ)
    {
      occ = occC;
      stage = cstage;
      fn = cstage ? (KernelFn)gi_dense_cta_kernel<3, true, false, 4> : (KernelFn)gi_dense_cta_kernel<3, false, false, 4>;
    }
  }
  LaunchCfg & c = s->cfg[0];
  c = LaunchCfg{};
  c.fn = fn;
  c.threads = threads;
  c.smem = stage ? smS : smN;
  c.occ = occ;
  c.stage = stage;
  c.lay = stage ? layS : layN;
  if(occ <= 0)
  {
    s->err = "problem does not fit in shared memory (n too large for the dense warp kernel)";
    return JRLQP_ERR_ARG;
  }
  cudaFuncAttributes attr;
  CK(cudaFuncGetAttributes(&attr, fn));
  c.regs = attr.numRegs;
  return JRLQP_OK;
}

// Warm calls. In automatic mode a warm layout of the shared-memory kernel that does not fit (n >= ~116: n (n - 1) / 2 more
// doubles than the cold one) sends the warm calls to the large-n kernel, which computes the same bits; cold calls keep the
// shared-memory kernel.
static int configure_warm(jrlqp_solver * s)
{
  if(s->cfg[1].fn) return JRLQP_OK;
  if(s->cfg[0].large) return use_large(s, true);
  const DenseSmem lay = make_layout(s->n, s->mc, s->nb, s->warps, false, true);
  const int smem = lay.total_doubles * 8;
  KernelFn fn = pick_warm_kernel(s->warps);
  if(smem > s->max_smem_optin && s->path_mode == 0) return use_large(s, true);
  if(!fn || smem > s->max_smem_optin)
  {
    s->err = "warm start: problem does not fit in shared memory (n too large; the Householder vectors need n (n - 1) / 2 more doubles)";
    return JRLQP_ERR_ARG;
  }
  const int occ = resident_ctas(s, fn, 32 * s->warps, smem);
  if(occ < 1)
  {
    s->err = "warm start kernel cannot be made resident";
    return JRLQP_ERR_ARG;
  }
  LaunchCfg & c = s->cfg[1];
  c = LaunchCfg{};
  c.threads = 32 * s->warps;
  c.smem = smem;
  c.occ = occ;
  c.lay = lay;
  c.fn = fn;
  return JRLQP_OK;
}

extern "C"
{

int jrlqp_version(void)
{
  return JRLQP_B200_VERSION;
}

void jrlqp_default_options(jrlqp_options * opt)
{
  opt->max_iter = 500;
  opt->big_bnd = 1e100;
  opt->warm_start = 0;
  opt->log_flags = 0;
}

int jrlqp_create(jrlqp_solver ** out, int32_t n, int32_t mc, int32_t use_bounds, int64_t batch_capacity, int32_t device)
{
  if(!out) return JRLQP_ERR_ARG;
  *out = nullptr;
  if(n < 1 || n > 1024 || mc < 0 || batch_capacity < 0) return JRLQP_ERR_ARG;
  jrlqp_solver * s = new jrlqp_solver();
  s->n = n;
  s->mc = mc;
  s->nb = use_bounds ? n : 0;
  s->m = mc + s->nb;
  s->capacity = batch_capacity;
  s->device = device;
  s->warps = std::min((n + 31) / 32, 4);
  jrlqp_default_options(&s->opt);
  *out = s; // returned even on CUDA failure so that jrlqp_last_error is readable
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if(device < 0 || device >= ndev)
  {
    s->err = "no such CUDA device";
    return JRLQP_ERR_CUDA;
  }
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if(prop.major != 10)
  {
    s->err = "this library contains sm_100a code only (Blackwell B200 required)";
    return JRLQP_ERR_CUDA;
  }
  {
    const char * e = getenv("JRLQP_SEQ_FCACHE");
    g_seq_fcache = e ? e[0] != '0' : 1;
  }
  if(const char * e = getenv("JRLQP_G_ZEROCOPY")) g_zero_copy_G = e[0] == '1' ? 1 : (e[0] == '0' ? 0 : -1);
  if(const char * e = getenv("JRLQP_H2D_FULL_G")) g_h2d_lower = !(e[0] == '1'); // tuning comparison: upload all of G
  s->num_sms = prop.multiProcessorCount;
  s->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  int rc = configure_kernel(s);
  if(rc != JRLQP_OK) return rc;
  CK(cudaMalloc(&s->d_counters, sizeof(unsigned long long) * kMaxChunks));
  CK(cudaMemset(s->d_counters, 0, sizeof(unsigned long long) * kMaxChunks));
#ifdef JRLQP_PHASE_TIMING
  CK(cudaMalloc(&s->d_phase, sizeof(unsigned long long) * 64));
  CK(cudaMemset(s->d_phase, 0, sizeof(unsigned long long) * 64));
#endif
  for(int i = 0; i < kStreams; ++i) CK(cudaStreamCreateWithFlags(&s->streams[i], cudaStreamNonBlocking));
  return JRLQP_OK;
}

int jrlqp_destroy(jrlqp_solver * s)
{
  if(!s) return JRLQP_OK;
  cudaSetDevice(s->device);
  void * ptrs[] = {s->d_fcache, s->d_cts, s->d_pre, s->d_pre_ok, s->d_ct, s->d_ct_busy, s->d_seq_it, s->d_seq_status, s->d_seq, s->d_seq_tot, s->large_cfg[0].work, s->large_cfg[1].work, s->large_cfg[0].busy, s->large_cfg[1].busy, s->d_as, s->d_phase, s->d_counters, s->d_G, s->d_a, s->d_C, s->d_bl, s->d_bu, s->d_xl, s->d_xu, s->d_x, s->d_u, s->d_f, s->d_L,
                   s->d_it, s->d_status, s->d_alist, s->d_nact, s->d_act};
  for(void * p : ptrs)
    if(p) cudaFree(p);
  for(int i = 0; i < kStreams; ++i)
    if(s->streams[i]) cudaStreamDestroy(s->streams[i]);
  if(s->ev_shared) cudaEventDestroy(s->ev_shared);
  if(s->ev_last) cudaEventDestroy(s->ev_last);
  delete s;
  return JRLQP_OK;
}

int jrlqp_set_options(jrlqp_solver * s, const jrlqp_options * opt)
{
  if(!s || !opt) return JRLQP_ERR_ARG;
  s->opt = *opt;
  return JRLQP_OK;
}

int jrlqp_get_options(const jrlqp_solver * s, jrlqp_options * opt)
{
  if(!s || !opt) return JRLQP_ERR_ARG;
  *opt = s->opt;
  return JRLQP_OK;
}

int jrlqp_set_stage_c(jrlqp_solver * s, int32_t mode)
{
  if(!s || mode < -1 || mode > 1) return JRLQP_ERR_ARG;
  s->stage_mode = mode;
  cudaSetDevice(s->device);
  return configure_kernel(s);
}

int jrlqp_set_kernel_path(jrlqp_solver * s, int32_t mode)
{
  if(!s || mode < 0 || mode > 2) return JRLQP_ERR_ARG;
  s->path_mode = mode;
  s->cfg[1] = LaunchCfg{};
  cudaSetDevice(s->device);
  return configure_kernel(s);
}

int64_t jrlqp_host_g_bytes(const jrlqp_solver * s, int32_t pinned)
{
  if(!s) return 0;
  const long long n = s->n, h = n / 2;
  if(pinned && !s->cfg[0].large && (g_zero_copy_G == 1 || (g_zero_copy_G < 0 && n <= 64))) return 8 * (n * (n + 1) / 2); // lower triangle, read in place
  if(g_h2d_lower && n >= 32) return 8 * (n * h + (n - h) * (n - h)); // left columns + bottom-right block
  return 8 * n * n;
}

int jrlqp_set_scan_transposed(jrlqp_solver * s, int32_t on)
{
  if(!s || on < -1 || on > 1) return JRLQP_ERR_ARG;
  s->scan_transposed = on;
  return JRLQP_OK;
}

int jrlqp_get_kernel_info(const jrlqp_solver * s, jrlqp_kernel_info * info)
{
  if(!s || !info) return JRLQP_ERR_ARG;
  const LaunchCfg & c = s->cfg[0];
  info->threads_per_qp = c.threads;
  info->rows_per_thread = c.large ? (s->n + kLargeThreads - 1) / kLargeThreads : 1;
  info->smem_bytes_per_qp = c.smem;
  info->qps_per_sm = c.occ;
  info->grid = c.occ * s->num_sms;
  info->num_sms = s->num_sms;
  info->stage_c = c.stage ? 1 : 0;
  info->regs_per_thread = c.regs;
  return JRLQP_OK;
}

/* Debug builds only (-DJRLQP_PHASE_TIMING): copies and clears the 4 x 16 per-warp, per-phase cycle
 * counters. Returns JRLQP_ERR_ARG in normal builds. Not declared in the public header. */
int jrlqp_debug_phase_cycles(jrlqp_solver * s, unsigned long long * out64)
{
  if(!s || !out64 || !s->d_phase) return JRLQP_ERR_ARG;
  CK(cudaSetDevice(s->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out64, s->d_phase, sizeof(unsigned long long) * 64, cudaMemcpyDeviceToHost));
  CK(cudaMemset(s->d_phase, 0, sizeof(unsigned long long) * 64));
  return JRLQP_OK;
}

int64_t jrlqp_launch_count(void)
{
  return g_launches.load();
}

const char * jrlqp_last_error(const jrlqp_solver * s)
{
  return s ? s->err.c_str() : "null solver";
}

static int validate(const jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res)
{
  if(!s || !pb || !res) return JRLQP_ERR_ARG;
  if(pb->batch < 0) return JRLQP_ERR_ARG;
  if(!pb->G || !pb->a || !res->x) return JRLQP_ERR_ARG;
  if(pb->ldg < s->n) return JRLQP_ERR_ARG;
  if(s->mc > 0 && (!pb->C || !pb->bl || !pb->bu || pb->ldc < s->n)) return JRLQP_ERR_ARG;
  if(s->nb > 0 && (!pb->xl || !pb->xu)) return JRLQP_ERR_ARG;
  if(s->nb == 0 && (pb->xl || pb->xu)) return JRLQP_ERR_ARG; // bounds given to a solver built without them
  return JRLQP_OK;
}

// Large-n kernel, G shared by the batch (stride 0): Cholesky and J = L^-T are computed ONCE, by one CTA running the
// solver's own factorisation code (same bits), and every solver CTA copies them instead of redoing 2/3 n^3 flops per
// instance (the MultiIK fixtures of config C spend ~100 % of a solve there). Asynchronous on `st`.
static bool uses_prefactor(const jrlqp_solver * s, const jrlqp_problem * pb, bool warm)
{
  return s->cfg[warm].large && pb->G_stride == 0 && pb->batch >= 2;
}

static int prefactor(jrlqp_solver * s, const jrlqp_problem * pb, cudaStream_t st)
{
  const long long n = s->n, ldl = (n + 3) & ~3ll, nv = ldl;
  if(!s->d_pre)
  {
    const LargeSmem lay(s->n, s->m, false);
    s->pre_smem = lay.total * 8;
    CK(jrlqp::raise_smem_limit(gi_large_prefactor_kernel<kLargeThreads>, s->pre_smem));
    CK(cudaMalloc(&s->d_pre, sizeof(double) * (size_t)(3 * n * ldl + 2 * nv)));
    CK(cudaMalloc(&s->d_pre_ok, sizeof(int)));
  }
  GiParams p{};
  p.n = s->n;
  p.mc = s->mc;
  p.nb = s->nb;
  p.ldg = pb->ldg;
  p.ldc = s->mc ? pb->ldc : s->n;
  p.batch = 1;
  p.G = pb->G;
  p.sG = 0;
  gi_large_prefactor_kernel<kLargeThreads><<<1, kLargeThreads, s->pre_smem, st>>>(p, s->d_pre, s->d_pre_ok);
  g_launches.fetch_add(1);
  CK(cudaGetLastError());
  return JRLQP_OK;
}

// Large-n kernel, C shared by the batch: one transposed copy per call for the coalesced constraint scan.
static bool uses_shared_ct(const jrlqp_solver * s, const jrlqp_problem * pb, bool warm)
{
  return s->cfg[warm].large && s->mc > 0 && pb->C_stride == 0 && pb->batch >= 2 && s->scan_transposed != 0;
}

static int prepare_shared_ct(jrlqp_solver * s, const jrlqp_problem * pb, cudaStream_t st)
{
  if(!s->d_cts)
  {
    s->ldcts = JRLQP_CT_LD;
    CK(cudaMalloc(&s->d_cts, sizeof(double) * (size_t)ct_doubles(s->n, s->mc)));
  }
  const dim3 grid((unsigned)((s->mc + 31) / 32), (unsigned)((s->n + 31) / 32));
  transpose_c_kernel<<<grid, 256, 0, st>>>(pb->C, pb->ldc, s->n, s->mc, s->d_cts);
  g_launches.fetch_add(1);
  CK(cudaGetLastError());
  return JRLQP_OK;
}

// measured (profiles/r01m_*): the transposed scan pays for wide CTAs (n = 128: +6 %), not for n = 50 (-4 %)
static bool scan_transposed_on(const jrlqp_solver * s)
{
  return s->scan_transposed != 0 && s->warps >= 3; // the narrow kernels (n <= 64) are compiled without it
}

// Slices for the transposed copy of C (gi_dense_cta.cuh: stage_ct): as many as CTAs of the shared-memory kernels
// (cold and warm, whatever the launch or stream) can be resident at the same time.
static int ensure_ct(jrlqp_solver * s)
{
  if(s->mc == 0 || !scan_transposed_on(s)) return JRLQP_OK;
  const int slots = 2 * std::max(s->cfg[0].occ, 1) * s->num_sms;
  if(s->d_ct && slots <= s->ct_slots) return JRLQP_OK;
  if(s->d_ct) CK(cudaFree(s->d_ct));
  if(s->d_ct_busy) CK(cudaFree(s->d_ct_busy));
  s->d_ct = nullptr;
  s->d_ct_busy = nullptr;
  s->ldct = JRLQP_CT_LD;
  s->ct_stride = (ct_doubles(s->n, s->mc) + 15) & ~15ll;
  s->ct_slots = slots;
  CK(cudaMalloc(&s->d_ct_busy, sizeof(int) * (size_t)slots));
  CK(cudaMemset(s->d_ct_busy, 0, sizeof(int) * (size_t)slots));
  CK(cudaMalloc(&s->d_ct, sizeof(double) * (size_t)s->ct_stride * (size_t)slots));
  return JRLQP_OK;
}

static int launch(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, cudaStream_t st, unsigned long long * counter, const CallArgs & call)
{
  const bool warm = call.warm;
  int rc = warm ? configure_warm(s) : JRLQP_OK;
  if(rc != JRLQP_OK) return rc;
  const LaunchCfg & cfg = s->cfg[warm];
  if(!cfg.large && (rc = ensure_ct(s)) != JRLQP_OK) return rc;
  GiParams p{};
  if(!cfg.large && s->mc > 0 && scan_transposed_on(s) && s->d_ct)
  {
    p.ct = s->d_ct;
    p.ct_stride = s->ct_stride;
    p.ct_busy = s->d_ct_busy;
    p.ct_slots = s->ct_slots;
    p.ldct = s->ldct;
  }
  p.n = s->n;
  p.mc = s->mc;
  p.nb = s->nb;
  p.ldg = pb->ldg;
  p.ldc = s->mc ? pb->ldc : s->n;
  p.batch = pb->batch;
  p.max_iter = s->opt.max_iter;
  p.big_bnd = s->opt.big_bnd;
  p.G = pb->G;
  p.sG = pb->G_stride;
  p.a = pb->a;
  p.sa = pb->a_stride;
  p.C = pb->C;
  p.sC = pb->C_stride;
  p.bl = pb->bl;
  p.sbl = pb->bl_stride;
  p.bu = pb->bu;
  p.sbu = pb->bu_stride;
  p.xl = pb->xl;
  p.sxl = pb->xl_stride;
  p.xu = pb->xu;
  p.sxu = pb->xu_stride;
  p.as_in = warm ? reinterpret_cast<const signed char *>(pb->as_in) : nullptr;
  p.s_as = pb->as_stride;
  p.warm_start = warm ? (call.force_warm_start ? 1 : s->opt.warm_start) : 0;
  p.x = res->x;
  p.u = res->u;
  p.f = res->f;
  p.iterations = res->iterations;
  p.status = res->status;
  p.active_set = res->active_set;
  p.active_list = res->active_list;
  p.n_active = res->n_active;
  p.L = res->L;
  p.counter = counter;
  p.phase_cycles = s->d_phase;
  p.lay = cfg.lay;
  p.fcache = s->d_fcache;
  p.fcache_stride = (long long)s->n * s->n + 2ll * s->n;
  p.fcache_mode = call.fcache_mode;
  p.work = cfg.work;
  p.work_stride = cfg.work_stride;
  p.work_busy = cfg.busy;
  p.work_slots = cfg.work_slots;
  p.ring_cols = cfg.ring_cols;
  p.slab_rows = cfg.slab_rows;
  long long grid = std::min<long long>((long long)cfg.occ * s->num_sms, std::max<long long>(pb->batch, 1));
  CK(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), st));
  if(uses_prefactor(s, pb, warm))
  {
    if(!call.pre_ready && (rc = prefactor(s, pb, st)) != JRLQP_OK) return rc;
    p.pre = s->d_pre;
    p.pre_ok = s->d_pre_ok;
  }
  if(uses_shared_ct(s, pb, warm))
  {
    if(!call.pre_ready && (rc = prepare_shared_ct(s, pb, st)) != JRLQP_OK) return rc;
    p.ct = s->d_cts;
    p.ldct = s->ldcts;
  }
  cfg.fn<<<(unsigned)grid, cfg.threads, cfg.smem, st>>>(p);
  g_launches.fetch_add(1);
  CK(cudaGetLastError());
  return JRLQP_OK;
}

// One in-flight device call per handle: a call enqueued on another stream than the previous one waits for it (event),
// calls on the same stream are ordered by the stream itself.
static int serialise_begin(jrlqp_solver * s, cudaStream_t st)
{
  if(s->has_last && st != s->last_stream) CK(cudaStreamWaitEvent(st, s->ev_last, 0));
  return JRLQP_OK;
}
static int serialise_end(jrlqp_solver * s, cudaStream_t st)
{
  if(!s->ev_last) CK(cudaEventCreateWithFlags(&s->ev_last, cudaEventDisableTiming));
  CK(cudaEventRecord(s->ev_last, st));
  s->last_stream = st;
  s->has_last = true;
  return JRLQP_OK;
}

int jrlqp_solve_batch_warm_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, void * stream)
{
  int rc = validate(s, pb, res);
  if(rc != JRLQP_OK) return rc;
  if(pb->batch == 0) return JRLQP_OK;
  CK(cudaSetDevice(s->device));
  unsigned long long * counter = s->d_counters + (s->next_counter++ % kMaxChunks);
  if((rc = serialise_begin(s, (cudaStream_t)stream)) != JRLQP_OK) return rc;
  rc = launch(s, pb, res, (cudaStream_t)stream, counter, CallArgs{true});
  if(rc != JRLQP_OK) return rc;
  return serialise_end(s, (cudaStream_t)stream);
}

int jrlqp_solve_batch_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, void * stream)
{
  int rc = validate(s, pb, res);
  if(rc != JRLQP_OK) return rc;
  if(pb->batch == 0) return JRLQP_OK;
  CK(cudaSetDevice(s->device));
  unsigned long long * counter = s->d_counters + (s->next_counter++ % kMaxChunks);
  if((rc = serialise_begin(s, (cudaStream_t)stream)) != JRLQP_OK) return rc;
  rc = launch(s, pb, res, (cudaStream_t)stream, counter, CallArgs{});
  if(rc != JRLQP_OK) return rc;
  return serialise_end(s, (cudaStream_t)stream);
}

// Device staging of the host entry point. Inputs shared by the whole batch (stride 0) take ONE slot, so a
// shared 387 x 387 Hessian with a 256k batch capacity costs 1.2 MB, not 300 GB; the buffers only grow.
static int ensure_buffer(jrlqp_solver * s, double ** buf, long long * cap, long long count, long long per)
{
  if(count <= *cap) return JRLQP_OK;
  if(*buf) CK(cudaFree(*buf));
  *buf = nullptr;
  *cap = 0;
  CK(cudaMalloc(buf, sizeof(double) * (size_t)std::max<long long>(count * per, 1)));
  *cap = count;
  return JRLQP_OK;
}

static int ensure_staging(jrlqp_solver * s, const jrlqp_problem * pb, bool wantL)
{
  const long long B = std::max<long long>(s->capacity, 1);
  const long long n = s->n, mc = s->mc, m = s->m;
  auto cnt = [&](long long stride) { return stride == 0 ? 1ll : B; };
  int rc;
  if((rc = ensure_buffer(s, &s->d_G, &s->cap_G, cnt(pb->G_stride), n * n)) != JRLQP_OK) return rc;
  if((rc = ensure_buffer(s, &s->d_a, &s->cap_a, cnt(pb->a_stride), n)) != JRLQP_OK) return rc;
  if(mc)
  {
    if((rc = ensure_buffer(s, &s->d_C, &s->cap_C, cnt(pb->C_stride), mc * n)) != JRLQP_OK) return rc;
    if((rc = ensure_buffer(s, &s->d_bl, &s->cap_bl, cnt(pb->bl_stride), mc)) != JRLQP_OK) return rc;
    if((rc = ensure_buffer(s, &s->d_bu, &s->cap_bu, cnt(pb->bu_stride), mc)) != JRLQP_OK) return rc;
  }
  if(s->nb)
  {
    if((rc = ensure_buffer(s, &s->d_xl, &s->cap_xl, cnt(pb->xl_stride), n)) != JRLQP_OK) return rc;
    if((rc = ensure_buffer(s, &s->d_xu, &s->cap_xu, cnt(pb->xu_stride), n)) != JRLQP_OK) return rc;
  }
  if(!s->staging_ready)
  {
    CK(cudaMalloc(&s->d_x, sizeof(double) * B * n));
    CK(cudaMalloc(&s->d_u, sizeof(double) * B * std::max<long long>(m, 1)));
    CK(cudaMalloc(&s->d_f, sizeof(double) * B));
    CK(cudaMalloc(&s->d_it, sizeof(int) * B));
    CK(cudaMalloc(&s->d_status, sizeof(int) * B));
    CK(cudaMalloc(&s->d_alist, sizeof(int) * B * n));
    CK(cudaMalloc(&s->d_nact, sizeof(int) * B));
    CK(cudaMalloc(&s->d_act, std::max<long long>(B * m, 1)));
    s->staging_ready = true;
  }
  if(wantL && !s->d_L) CK(cudaMalloc(&s->d_L, sizeof(double) * B * n * n));
  return JRLQP_OK;
}

// Copy `count` instances of a (possibly strided, possibly ld-padded) host array into the dense
// device staging buffer. rows x cols column-major blocks with leading dimension ld.
static cudaError_t h2d(double * dst, const double * src, long long stride, long long count, int rows, int cols, int ld, cudaStream_t st)
{
  const long long blk = (long long)rows * cols;
  if(stride == 0) count = 1;
  if(ld == rows && (stride == blk || count == 1)) return cudaMemcpyAsync(dst, src, sizeof(double) * blk * count, cudaMemcpyHostToDevice, st);
  if(ld == rows) return cudaMemcpy2DAsync(dst, sizeof(double) * blk, src, sizeof(double) * stride, sizeof(double) * blk, count, cudaMemcpyHostToDevice, st);
  for(long long k = 0; k < count; ++k)
  {
    cudaError_t e = cudaMemcpy2DAsync(dst + k * blk, sizeof(double) * rows, src + k * stride, sizeof(double) * ld, sizeof(double) * rows, cols,
                                      cudaMemcpyHostToDevice, st);
    if(e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// Upload of G for the host entry points: the kernels read the lower triangle only (as the reference's LLT does,
// src/GoldfarbIdnaniSolver.cpp:58), so the top-right (n/2) x (n - n/2) block of every instance need not cross PCIe:
// the left n/2 columns go as one contiguous piece per instance (2-D copy), the bottom-right block as a 3-D copy
// (rows of n - n/2 doubles). 25 % of G = 11.5 % of the input bytes of the headline shape. Falls back to the plain
// copy when the layout is not the dense one or the blocks would be too small to be worth two descriptors.
static cudaError_t h2d_G(double * dst, const double * src, long long stride, long long count, int n, int ld, cudaStream_t st)
{
  const int h = n / 2;
  if(!g_h2d_lower || stride == 0 || count < 64 || ld != n || n < 32 || stride % n != 0) return h2d(dst, src, stride, count, n, n, ld, st);
  cudaError_t e = cudaMemcpy2DAsync(dst, sizeof(double) * (size_t)n * n, src, sizeof(double) * (size_t)stride, sizeof(double) * (size_t)h * n,
                                    (size_t)count, cudaMemcpyHostToDevice, st);
  if(e != cudaSuccess) return e;
  cudaMemcpy3DParms p3{};
  p3.srcPtr = make_cudaPitchedPtr(const_cast<double *>(src), sizeof(double) * (size_t)n, sizeof(double) * (size_t)n, (size_t)(stride / n));
  p3.dstPtr = make_cudaPitchedPtr(dst, sizeof(double) * (size_t)n, sizeof(double) * (size_t)n, (size_t)n);
  p3.srcPos = make_cudaPos(sizeof(double) * (size_t)h, (size_t)h, 0);
  p3.dstPos = make_cudaPos(sizeof(double) * (size_t)h, (size_t)h, 0);
  p3.extent = make_cudaExtent(sizeof(double) * (size_t)(n - h), (size_t)(n - h), (size_t)count);
  p3.kind = cudaMemcpyHostToDevice;
  return cudaMemcpy3DAsync(&p3, st);
}

enum : int
{
  kStageShared = 1, // arrays shared by the batch (stride 0): one slot each
  kStageInstances = 2 // the other arrays, and as_in
};

// Fills `dp` with the device copy, in the handle's staging, of instances [b0, b0 + cnt) of the caller's host problem `pb`,
// and enqueues on `st` the copies of the arrays `which` selects. Arrays left null in `pb` are not staged. G crosses whole,
// or in the two-block layout of h2d_G with `lower_G`, or not at all when `mapped_G` (the device alias of the caller's
// pinned G, read in place by the kernels) is given.
static int stage_host_problem(jrlqp_solver * s, const jrlqp_problem * pb, long long b0, long long cnt, int which, bool lower_G,
                              const double * mapped_G, cudaStream_t st, jrlqp_problem * dp)
{
  const long long n = s->n, mc = s->mc, m = s->m;
  auto up = [&](double * dbase, const double * h, long long hstride, int rows, int cols, int ld, const double *& dptr, int64_t & dstride,
                bool lower = false) -> cudaError_t
  {
    if(!h) return cudaSuccess;
    const long long blk = (long long)rows * cols;
    double * d = hstride == 0 ? dbase : dbase + b0 * blk;
    dptr = d;
    dstride = hstride == 0 ? 0 : blk;
    if(!(which & (hstride == 0 ? kStageShared : kStageInstances))) return cudaSuccess;
    return lower ? h2d_G(d, h + b0 * hstride, hstride, cnt, rows, ld, st) : h2d(d, h + b0 * hstride, hstride, cnt, rows, cols, ld, st);
  };
  dp->batch = cnt;
  if(mapped_G)
  {
    dp->G = mapped_G + b0 * pb->G_stride;
    dp->G_stride = pb->G_stride;
  }
  else
    CK(up(s->d_G, pb->G, pb->G_stride, (int)n, (int)n, pb->ldg, dp->G, dp->G_stride, lower_G));
  dp->ldg = mapped_G ? pb->ldg : (int)n;
  CK(up(s->d_a, pb->a, pb->a_stride, (int)n, 1, (int)n, dp->a, dp->a_stride));
  if(mc)
  {
    CK(up(s->d_C, pb->C, pb->C_stride, (int)n, (int)mc, pb->ldc, dp->C, dp->C_stride));
    CK(up(s->d_bl, pb->bl, pb->bl_stride, (int)mc, 1, (int)mc, dp->bl, dp->bl_stride));
    CK(up(s->d_bu, pb->bu, pb->bu_stride, (int)mc, 1, (int)mc, dp->bu, dp->bu_stride));
  }
  dp->ldc = (int)n;
  if(s->nb)
  {
    CK(up(s->d_xl, pb->xl, pb->xl_stride, (int)n, 1, (int)n, dp->xl, dp->xl_stride));
    CK(up(s->d_xu, pb->xu, pb->xu_stride, (int)n, 1, (int)n, dp->xu, dp->xu_stride));
  }
  if(pb->as_in && (which & kStageInstances))
  {
    if(!s->d_as) CK(cudaMalloc(&s->d_as, std::max<long long>(std::max<long long>(s->capacity, 1) * m, 1)));
    const long long cnt_as = pb->as_stride == 0 ? 1 : cnt;
    signed char * das = s->d_as + b0 * m;
    if(pb->as_stride == m || cnt_as == 1)
      CK(cudaMemcpyAsync(das, pb->as_in + b0 * pb->as_stride, (size_t)(cnt_as * m), cudaMemcpyHostToDevice, st));
    else
      CK(cudaMemcpy2DAsync(das, (size_t)m, pb->as_in + b0 * pb->as_stride, (size_t)pb->as_stride, (size_t)m, (size_t)cnt_as, cudaMemcpyHostToDevice, st));
    dp->as_in = reinterpret_cast<const int8_t *>(das);
    dp->as_stride = pb->as_stride == 0 ? 0 : m;
  }
  return JRLQP_OK;
}

static int solve_batch_host_impl(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res, bool warm)
{
  int rc = validate(s, pb, res);
  if(rc != JRLQP_OK) return rc;
  if(pb->batch > s->capacity) return JRLQP_ERR_CAPACITY;
  if(pb->batch == 0) return JRLQP_SUCCESS;
  CK(cudaSetDevice(s->device));
  rc = ensure_staging(s, pb, res->L != nullptr);
  if(rc != JRLQP_OK) return rc;
  if(warm && (rc = configure_warm(s)) != JRLQP_OK) return rc;

  const long long B = pb->batch;
  const long long n = s->n, mc = s->mc, m = s->m;
  // Where the host link bounds the call (small n: 43 KB of input per n = 50 QP against a solve of 0.5 us per QP and
  // GPU), the kernels read G straight from the caller's PINNED buffer: only the lower triangle crosses PCIe, as
  // SM-initiated reads concurrent with the DMA of the other arrays (measured, profiles/r01u_*: +5 % at n = 50, +9 % at
  // n = 20 over the two-block upload, -5 % at n = 128, which is kernel-bound: automatic mode = n <= 64).
  const bool zero_copy_G = !s->cfg[warm].large && !res->L && pb->G_stride != 0 && (g_zero_copy_G == 1 || (g_zero_copy_G < 0 && s->n <= 64));
  const double * g_dev_ptr_G = nullptr;
  if(zero_copy_G)
  {
    cudaPointerAttributes at{};
    if(cudaPointerGetAttributes(&at, pb->G) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer != nullptr)
      g_dev_ptr_G = static_cast<const double *>(at.devicePointer);
    else
      cudaGetLastError();
  }
  // Pipeline: split the batch into chunks; chunk c runs H2D -> kernel -> D2H on stream c % kStreams,
  // so the copy engines and the SMs overlap across chunks.
  const long long per_qp_bytes = 8 * (n * n + n + mc * n + 2 * mc + 2 * s->nb);
  long long chunk = std::max<long long>((long long)s->cfg[0].occ * s->num_sms * 4, (48ll << 20) / std::max<long long>(per_qp_bytes, 1));
  long long nchunks = std::min<long long>(kMaxChunks, std::max<long long>(1, (B + chunk - 1) / chunk));
  if(const char * e = getenv("JRLQP_HOST_CHUNK")) // tuning: QPs per chunk of the host pipeline (scripts/e2e_chunk_sweep.py)
  {
    const long long v = atoll(e);
    if(v > 0) nchunks = std::min<long long>(kMaxChunks, std::max<long long>(1, (B + v - 1) / v));
  }
  chunk = (B + nchunks - 1) / nchunks;

  jrlqp_problem hp = *pb;
  if(!warm) hp.as_in = nullptr; // (read by warm calls only)
  const bool lower_G = !res->L; // (the factor copy-out reads nothing of G's upper part either, but keep it simple)
  // arrays shared by the batch (stride 0): uploaded once, on stream 0, with the factor of a shared G and the transposed copy
  // of a shared C that all the chunks re-use; the other streams wait for them
  if(pb->G_stride == 0 || pb->a_stride == 0 || (mc && (pb->C_stride == 0 || pb->bl_stride == 0 || pb->bu_stride == 0))
     || (s->nb && (pb->xl_stride == 0 || pb->xu_stride == 0)))
  {
    jrlqp_problem dsh{};
    if((rc = stage_host_problem(s, &hp, 0, B, kStageShared, lower_G, g_dev_ptr_G, s->streams[0], &dsh)) != JRLQP_OK) return rc;
    if(uses_prefactor(s, &dsh, warm) && (rc = prefactor(s, &dsh, s->streams[0])) != JRLQP_OK) return rc;
    if(uses_shared_ct(s, &dsh, warm) && (rc = prepare_shared_ct(s, &dsh, s->streams[0])) != JRLQP_OK) return rc;
    if(!s->ev_shared) CK(cudaEventCreateWithFlags(&s->ev_shared, cudaEventDisableTiming));
    CK(cudaEventRecord(s->ev_shared, s->streams[0]));
    for(int i = 1; i < kStreams; ++i) CK(cudaStreamWaitEvent(s->streams[i], s->ev_shared, 0));
  }

  for(long long c = 0; c < nchunks; ++c)
  {
    const long long b0 = c * chunk;
    const long long cnt = std::min(chunk, B - b0);
    if(cnt <= 0) break;
    cudaStream_t st = s->streams[c % kStreams];
    jrlqp_problem dp{};
    if((rc = stage_host_problem(s, &hp, b0, cnt, kStageInstances, lower_G, g_dev_ptr_G, st, &dp)) != JRLQP_OK) return rc;
    jrlqp_result dr{};
    dr.x = s->d_x + b0 * n;
    dr.u = res->u ? s->d_u + b0 * m : nullptr;
    dr.f = res->f ? s->d_f + b0 : nullptr;
    dr.iterations = res->iterations ? s->d_it + b0 : nullptr;
    dr.status = s->d_status + b0;
    dr.active_set = res->active_set ? s->d_act + b0 * m : nullptr;
    dr.active_list = res->active_list ? s->d_alist + b0 * n : nullptr;
    dr.n_active = res->n_active ? s->d_nact + b0 : nullptr;
    dr.L = res->L ? s->d_L + b0 * n * n : nullptr;
    rc = launch(s, &dp, &dr, st, s->d_counters + (c % kMaxChunks), CallArgs{warm, false, /*pre_ready=*/true}); // shared factor / transposed C prepared above
    if(rc != JRLQP_OK) return rc;
    CK(cudaMemcpyAsync(res->x + b0 * n, dr.x, sizeof(double) * cnt * n, cudaMemcpyDeviceToHost, st));
    if(res->u && m) CK(cudaMemcpyAsync(res->u + b0 * m, dr.u, sizeof(double) * cnt * m, cudaMemcpyDeviceToHost, st));
    if(res->f) CK(cudaMemcpyAsync(res->f + b0, dr.f, sizeof(double) * cnt, cudaMemcpyDeviceToHost, st));
    if(res->iterations) CK(cudaMemcpyAsync(res->iterations + b0, dr.iterations, sizeof(int) * cnt, cudaMemcpyDeviceToHost, st));
    if(res->status) CK(cudaMemcpyAsync(res->status + b0, dr.status, sizeof(int) * cnt, cudaMemcpyDeviceToHost, st));
    if(res->active_set && m) CK(cudaMemcpyAsync(res->active_set + b0 * m, dr.active_set, cnt * m, cudaMemcpyDeviceToHost, st));
    if(res->active_list) CK(cudaMemcpyAsync(res->active_list + b0 * n, dr.active_list, sizeof(int) * cnt * n, cudaMemcpyDeviceToHost, st));
    if(res->n_active) CK(cudaMemcpyAsync(res->n_active + b0, dr.n_active, sizeof(int) * cnt, cudaMemcpyDeviceToHost, st));
    if(res->L) CK(cudaMemcpyAsync(res->L + b0 * n * n, dr.L, sizeof(double) * cnt * n * n, cudaMemcpyDeviceToHost, st));
  }
  for(int i = 0; i < kStreams; ++i) CK(cudaStreamSynchronize(s->streams[i]));

  // worst status of the batch (the reference's return value, reduced over the batch)
  int worst = 0;
  if(res->status)
  {
    for(long long b = 0; b < B; ++b) worst = std::max(worst, res->status[b]);
  }
  else
  {
    std::vector<int> hs((size_t)B);
    CK(cudaMemcpy(hs.data(), s->d_status, sizeof(int) * B, cudaMemcpyDeviceToHost));
    for(long long b = 0; b < B; ++b) worst = std::max(worst, hs[(size_t)b]);
  }
  return worst;
}

int jrlqp_solve_batch_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res)
{
  return solve_batch_host_impl(s, pb, res, false);
}

int jrlqp_solve_batch_warm_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_result * res)
{
  return solve_batch_host_impl(s, pb, res, true);
}

// ---------------------------------------------------------------------------------------------
// Warm-started sequences (benchmarks/SolversWarmStart.cpp:234-276)
// ---------------------------------------------------------------------------------------------
__global__ void seq_accumulate_kernel(const int * __restrict__ it, const int * __restrict__ status, int * it_total, int * status_worst, long long batch, int first)
{
  const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if(b >= batch) return;
  if(it_total) it_total[b] = (first ? 0 : it_total[b]) + it[b];
  if(status_worst) status_worst[b] = first ? status[b] : max(status_worst[b], status[b]);
}

static int validate_sequence(const jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res, bool device)
{
  int rc = validate(s, pb, res);
  if(rc != JRLQP_OK) return rc;
  if(!seq || seq->steps < 1) return JRLQP_ERR_ARG;
  if(device && seq->warm && !res->active_set) return JRLQP_ERR_ARG; // carries the active set from step to step
  return JRLQP_OK;
}

static int sequence_device_impl(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res, cudaStream_t st)
{
  const long long B = pb->batch;
  const bool totals = seq->iterations_total || seq->status_worst;
  if(totals && (!res->iterations || !res->status) && B > s->cap_seq)
  {
    if(s->d_seq_it) CK(cudaFree(s->d_seq_it));
    if(s->d_seq_status) CK(cudaFree(s->d_seq_status));
    s->d_seq_it = s->d_seq_status = nullptr;
    s->cap_seq = 0;
    CK(cudaMalloc(&s->d_seq_it, sizeof(int) * (size_t)B));
    CK(cudaMalloc(&s->d_seq_status, sizeof(int) * (size_t)B));
    s->cap_seq = B;
  }
  if(seq->warm)
  {
    int rc = configure_warm(s);
    if(rc != JRLQP_OK) return rc;
  }
  // G is the same at every step: the warm kernels keep the factor of step 0 in HBM and re-read it afterwards (same bits)
  const bool use_fcache = seq->warm != 0 && !s->cfg[1].large && seq->steps > 1 && !res->L && g_seq_fcache != 0;
  if(use_fcache)
  {
    const long long need = B * ((long long)s->n * s->n + 2ll * s->n);
    if(need > s->fcache_cap)
    {
      if(s->d_fcache) CK(cudaFree(s->d_fcache));
      s->d_fcache = nullptr;
      s->fcache_cap = 0;
      if(cudaMalloc(&s->d_fcache, sizeof(double) * (size_t)need) == cudaSuccess)
        s->fcache_cap = need;
      else
        cudaGetLastError(); // (no room: the steps factorise again, as before)
    }
  }
  unsigned long long * counter = s->d_counters + (s->next_counter++ % kMaxChunks);
  for(int t = 0; t < seq->steps; ++t)
  {
    const int fcache_mode = (use_fcache && s->d_fcache != nullptr && B * ((long long)s->n * s->n + 2ll * s->n) <= s->fcache_cap) ? (t == 0 ? 1 : 2) : 0;
    jrlqp_problem p = *pb;
    p.a = pb->a + (long long)t * seq->a_step_stride;
    jrlqp_result r = *res;
    r.x = res->x + (long long)t * seq->x_step_stride;
    if(res->u) r.u = res->u + (long long)t * seq->u_step_stride;
    if(res->f) r.f = res->f + (long long)t * seq->f_step_stride;
    if(res->iterations) r.iterations = res->iterations + (long long)t * seq->iterations_step_stride;
    if(res->status) r.status = res->status + (long long)t * seq->status_step_stride;
    if(totals)
    {
      if(!r.iterations) r.iterations = s->d_seq_it;
      if(!r.status) r.status = s->d_seq_status;
    }
    if(seq->warm && t > 0)
    {
      // the active set the previous step ended with, read in place: an instance reads its guess
      // when it starts and writes its final set when it ends, and no other CTA touches that row
      p.as_in = res->active_set;
      p.as_stride = s->m;
    }
    int rc = launch(s, &p, &r, st, counter, CallArgs{seq->warm != 0, seq->warm != 0, /*pre_ready=*/t > 0, fcache_mode});
    if(rc != JRLQP_OK) return rc;
    if(totals)
    {
      const unsigned grid = (unsigned)((B + 255) / 256);
      seq_accumulate_kernel<<<grid, 256, 0, st>>>(r.iterations, r.status, seq->iterations_total, seq->status_worst, B, t == 0);
      g_launches.fetch_add(1);
      CK(cudaGetLastError());
    }
  }
  return JRLQP_OK;
}

int jrlqp_solve_sequence_device(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res, void * stream)
{
  int rc = validate_sequence(s, pb, seq, res, true);
  if(rc != JRLQP_OK) return rc;
  if(pb->batch == 0) return JRLQP_OK;
  CK(cudaSetDevice(s->device));
  if((rc = serialise_begin(s, (cudaStream_t)stream)) != JRLQP_OK) return rc;
  rc = sequence_device_impl(s, pb, seq, res, (cudaStream_t)stream);
  if(rc != JRLQP_OK) return rc;
  return serialise_end(s, (cudaStream_t)stream);
}

int jrlqp_solve_sequence_host(jrlqp_solver * s, const jrlqp_problem * pb, const jrlqp_sequence * seq, const jrlqp_result * res)
{
  int rc = validate_sequence(s, pb, seq, res, false);
  if(rc != JRLQP_OK) return rc;
  if(pb->batch > s->capacity) return JRLQP_ERR_CAPACITY;
  if(pb->batch == 0) return JRLQP_SUCCESS;
  if(res->L) return JRLQP_ERR_ARG; // the factor does not change along a sequence: ask one plain solve for it
  CK(cudaSetDevice(s->device));
  rc = ensure_staging(s, pb, false);
  if(rc != JRLQP_OK) return rc;
  const long long B = pb->batch, n = s->n, m = s->m, T = seq->steps;
  cudaStream_t st = s->streams[0];
  // arena: [T][B][n] linear terms, then the per-step outputs that were asked for
  const long long na = T * B * n;
  const long long nx = seq->x_step_stride ? T * B * n : 0;
  const long long nu = (res->u && seq->u_step_stride) ? T * B * std::max<long long>(m, 1) : 0;
  const long long nf = (res->f && seq->f_step_stride) ? T * B : 0;
  const long long ni = (res->iterations && seq->iterations_step_stride) ? (T * B + 1) / 2 : 0; // ints, packed in doubles
  const long long ns = (res->status && seq->status_step_stride) ? (T * B + 1) / 2 : 0;
  const long long need = na + nx + nu + nf + ni + ns;
  if(need > s->cap_seq_arena)
  {
    if(s->d_seq) CK(cudaFree(s->d_seq));
    s->d_seq = nullptr;
    s->cap_seq_arena = 0;
    CK(cudaMalloc(&s->d_seq, sizeof(double) * (size_t)need));
    s->cap_seq_arena = need;
  }
  if(!s->d_seq_tot) CK(cudaMalloc(&s->d_seq_tot, sizeof(int) * 2 * (size_t)std::max<long long>(s->capacity, 1)));
  double * d_aseq = s->d_seq;
  double * d_xs = d_aseq + na;
  double * d_us = d_xs + nx;
  double * d_fs = d_us + nu;
  int * d_is = reinterpret_cast<int *>(d_fs + nf);
  int * d_ss = reinterpret_cast<int *>(d_fs + nf + ni);

  jrlqp_problem hp = *pb;
  hp.a = nullptr; // (the linear terms of every step go to the arena, below)
  if(!seq->warm) hp.as_in = nullptr;
  jrlqp_problem dp{};
  if((rc = stage_host_problem(s, &hp, 0, B, kStageShared | kStageInstances, false, nullptr, st, &dp)) != JRLQP_OK) return rc;
  // linear terms: step t, instance b at a + t * a_step_stride + b * a_stride  ->  dense [T][B][n]
  for(long long t = 0; t < T; ++t)
  {
    const double * h = pb->a + t * seq->a_step_stride;
    if(pb->a_stride == 0)
      for(long long b = 0; b < B; ++b) CK(cudaMemcpyAsync(d_aseq + (t * B + b) * n, h, sizeof(double) * n, cudaMemcpyHostToDevice, st)); // shared within a step (rare)
    else
      CK(h2d(d_aseq + t * B * n, h, pb->a_stride, B, (int)n, 1, (int)n, st));
  }
  dp.a = d_aseq;
  dp.a_stride = n;
  jrlqp_sequence ds = *seq;
  ds.a_step_stride = B * n;
  ds.x_step_stride = nx ? B * n : 0;
  ds.u_step_stride = nu ? B * m : 0;
  ds.f_step_stride = nf ? B : 0;
  ds.iterations_step_stride = ni ? B : 0;
  ds.status_step_stride = ns ? B : 0;
  ds.iterations_total = s->d_seq_tot;
  ds.status_worst = s->d_seq_tot + std::max<long long>(s->capacity, 1);
  jrlqp_result dr{};
  dr.x = nx ? d_xs : s->d_x;
  dr.u = res->u ? (nu ? d_us : s->d_u) : nullptr;
  dr.f = res->f ? (nf ? d_fs : s->d_f) : nullptr;
  dr.iterations = res->iterations ? (ni ? d_is : s->d_it) : nullptr;
  dr.status = res->status ? (ns ? d_ss : s->d_status) : nullptr;
  dr.active_set = (res->active_set || seq->warm) ? s->d_act : nullptr;
  dr.active_list = res->active_list ? s->d_alist : nullptr;
  dr.n_active = res->n_active ? s->d_nact : nullptr;
  rc = sequence_device_impl(s, &dp, &ds, &dr, st);
  if(rc != JRLQP_OK) return rc;
  // read back: per-step outputs step by step (the host strides are the caller's), the rest once
  auto down = [&](void * h, const void * d, long long hstep, long long dstep, size_t elem, long long per) -> cudaError_t
  {
    const long long steps = hstep ? T : 1;
    for(long long t = 0; t < steps; ++t)
    {
      cudaError_t e = cudaMemcpyAsync((char *)h + t * hstep * elem, (const char *)d + t * dstep * elem, elem * (size_t)(B * per), cudaMemcpyDeviceToHost, st);
      if(e != cudaSuccess) return e;
    }
    return cudaSuccess;
  };
  CK(down(res->x, dr.x, seq->x_step_stride, ds.x_step_stride, sizeof(double), n));
  if(res->u && m) CK(down(res->u, dr.u, seq->u_step_stride, ds.u_step_stride, sizeof(double), m));
  if(res->f) CK(down(res->f, dr.f, seq->f_step_stride, ds.f_step_stride, sizeof(double), 1));
  if(res->iterations) CK(down(res->iterations, dr.iterations, seq->iterations_step_stride, ds.iterations_step_stride, sizeof(int), 1));
  if(res->status) CK(down(res->status, dr.status, seq->status_step_stride, ds.status_step_stride, sizeof(int), 1));
  if(res->active_set && m) CK(cudaMemcpyAsync(res->active_set, dr.active_set, (size_t)(B * m), cudaMemcpyDeviceToHost, st));
  if(res->active_list) CK(cudaMemcpyAsync(res->active_list, dr.active_list, sizeof(int) * (size_t)(B * n), cudaMemcpyDeviceToHost, st));
  if(res->n_active) CK(cudaMemcpyAsync(res->n_active, dr.n_active, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, st));
  if(seq->iterations_total) CK(cudaMemcpyAsync(seq->iterations_total, ds.iterations_total, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, st));
  std::vector<int> worst((size_t)B);
  CK(cudaMemcpyAsync(worst.data(), ds.status_worst, sizeof(int) * (size_t)B, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if(seq->status_worst) std::memcpy(seq->status_worst, worst.data(), sizeof(int) * (size_t)B);
  int w = 0;
  for(long long b = 0; b < B; ++b) w = std::max(w, worst[(size_t)b]);
  return w;
}

} // extern "C"

#ifdef JRLQP_TEST_FALLBACKS
// Test build only (test_fallbacks.cuh): per-site counts of the fallbacks taken, and the flag that makes every proof decline.
// counts (HOST, 3 x FB_NSITES): the sites reached from this unit (dense and large kernels), from structured.cu (structured
// LLT and solves) and from blockgi.cu (BlockGI), in that order; the counters are cleared. Device 0.
namespace jrlqp
{
int fb_collect_structured(unsigned long long * out);
int fb_collect_blockgi(unsigned long long * out);
int fb_set_decline_structured(int on);
int fb_set_decline_blockgi(int on);
} // namespace jrlqp

extern "C" int jrlqp_test_fallback_counts(uint64_t * counts)
{
  unsigned long long * c = reinterpret_cast<unsigned long long *>(counts);
  for(int s = 0; s < 3 * jrlqp::FB_NSITES; ++s) c[s] = 0;
  int rc = jrlqp::fb_collect(c);
  if(rc == 0) rc = jrlqp::fb_collect_structured(c + jrlqp::FB_NSITES);
  if(rc == 0) rc = jrlqp::fb_collect_blockgi(c + 2 * jrlqp::FB_NSITES);
  return rc;
}

extern "C" int jrlqp_test_fallback_decline_all(int32_t on)
{
  int rc = jrlqp::fb_set_decline(on);
  if(rc == 0) rc = jrlqp::fb_set_decline_structured(on);
  if(rc == 0) rc = jrlqp::fb_set_decline_blockgi(on);
  return rc;
}
#endif
