// Structured dual active-set solver, batched: ONE QP PER CTA, persistent CTAs pulling problems from a
// ticket counter.
//
// Replaces, for a batch of QPs sharing one block structure, experimental::BlockGISolver::solve
// (src/experimental/BlockGISolver.cpp:18-60) and what it runs on:
//   DualSolver::solve                         src/DualSolver.cpp:91-168 (the loop), :231-244 (add / remove)
//   BlockGISolver::init_ and its helpers       src/experimental/BlockGISolver.cpp:62-109, 293-377, 454-484
//   selectViolatedConstraint_ / computeStep_ / computeStepLength_ / dot_   :111-275
//   structured::StructuredJ::premultByJt / premultByJ2   src/structured/StructuredJ.cpp:33-57
//   structured::StructuredQR::RSolve / add / remove      src/structured/StructuredQR.cpp:66-103
//   structured::StructuredC::col / transposeMult         src/structured/StructuredC.cpp:57-77
//   internal::OrthonormalSequence (Householder / Givens elements, both directions)
//                                                        src/internal/OrthonormalSequence.cpp:50-124,178-196
// The matrix J = L^-T Q of the dense solver is never formed: L is the structured Cholesky factor of G
// (structured.cuh, factorised by structured_llt_kernel before this kernel runs), Q the product of one
// Householder reflector per activated constraint and one Givens sequence per dropped one, kept as a
// growing list of records in a per-CTA slice of global memory (it stays in L2 for the sizes of the
// reference's use cases). One iteration costs O(n nb) for the two structured solves plus O(sum of record
// lengths) for the two passes over Q, instead of the O(n^2) of the dense solver.
//
// Mapping: vectors (x, z, d, u, r, one work vector), the active set and the record table live in shared
// memory; the structured solves use every thread of the CTA (tile by tile, structured.cuh); the passes
// over Q are one serial chain of short reflections (dot, scale, axpy over <= n elements), which ONE warp
// runs with shuffle reductions and no block barrier; constraint scan and ratio test are block-wide
// first-minimum reductions. Arithmetic: the canonical orders of oracle/block_oracle.hpp, so results are
// bit-identical to the CPU oracle.
#pragma once

#include "fp64_exact.cuh"
#include "structured.cuh"
#include "tri_warp_solve.cuh"

namespace jrlqp
{

// fast paths of the kernel (BlockGiParams::flags; all on by default, JRLQP_BLOCKGI_FAST overrides for A/B runs and tests)
enum : int
{
  BGF_WARP_SOLVE = 1, // structured solves on one warp, tiles streamed by TMA bulk copies (needs fast_nb != 0)
  BGF_REG_SEQUENCE = 2, // orthonormal sequence applied to a vector held in registers, one barrier per reflector
  BGF_BLOCKED_RSOLVE = 4 // R^-1 d1 blocked by 16 columns: register-resident triangle on one warp + panel update by the CTA
};

struct BlockGiParams
{
  StructParams G; // descriptor; data = the factorised blocks (instance k at data + k * stride; stride 0: shared)
  const int * llt_ok; // [batch] (or [1] when G is shared): 0 = not positive definite
  int ok_stride;
  // structured::StructuredC
  int cb;
  const int * cnvar; // [cb]
  const long long * coff; // [cb]
  const int * cld; // [cb]
  const int * cvar0; // [cb + 1] first variable of block i
  const int * ccstr0; // [cb + 1] first constraint of block i
  const int * toblock; // [mc]
  int mc, nb, max_iter;
  double big_bnd;
  const double *a, *C, *bl, *bu, *xl, *xu;
  long long sa, sC, sbl, sbu, sxl, sxu;
  double *x, *u, *f;
  int *iters, *status;
  signed char * act;
  int *alist, *nact;
  long long * qdoubles; // nullable: doubles of Q storage used (statistic)
  double * ws; // per-CTA workspace: R packed (n (n + 1) / 2), then the Q records (qcap)
  long long ws_stride, qcap;
  int fast_nb; // tile size of a tri-block-diagonal chain of uniform dense tiles at 16-byte aligned offsets (8 / 12 / 16), else 0
  int flags; // BGF_*
  long long batch;
  unsigned long long * ticket;
};

enum : int
{
  BG_INACTIVE = 0,
  BG_LOWER = 1,
  BG_UPPER = 2,
  BG_EQUALITY = 3,
  BG_LOWER_BOUND = 4,
  BG_UPPER_BOUND = 5,
  BG_FIXED = 6
};

#define BG_FULL 0xffffffffu

// Eigen JacobiRotation::makeGivens, real case (as gi_oracle.cpp makeGivens)
__device__ __forceinline__ void bg_make_givens(double p, double q, double & c, double & s, double & r)
{
  if(q == 0.0)
  {
    c = p < 0.0 ? -1.0 : 1.0;
    s = 0.0;
    r = fabs(p);
  }
  else if(p == 0.0)
  {
    c = 0.0;
    s = q < 0.0 ? 1.0 : -1.0;
    r = fabs(q);
  }
  else if(fabs(p) > fabs(q))
  {
    const double t = q / p;
    double u = sqrt(fma(t, t, 1.0));
    if(p < 0.0) u = -u;
    c = 1.0 / u;
    s = -t * c;
    r = p * u;
  }
  else
  {
    const double t = p / q;
    double u = sqrt(fma(t, t, 1.0));
    if(q < 0.0) u = -u;
    s = -1.0 / u;
    c = -t * s;
    r = q * u;
  }
}

// ME: entries of a reflector / of a vector per thread in the passes over Q (128 classes x ME >= n)
template<int ME>
struct BlockGi
{
  static constexpr int RING = TriWarp::RING; // stage of the warp-level structured solves (tri_warp_solve.cuh)
  static constexpr int QD = 3; // stage of the passes over Q: reflectors of QD records in flight (cp.async, thread-private slots)
  static constexpr int RB = 16; // columns per block of the blocked R solve
  const BlockGiParams & P;
  const int n, mc, m, T, tid, lane, warp, W;
  const bool up;
  // shared memory
  double *x, *z, *d, *w, *u, *r, *scr, *hred, *rtri, *qring, *rtau, *Lt, *Bt, *ring;
  int MJ; // entries of a vector per thread in the passes over Q: ceil(n / 128) <= ME
  double2 * dgp; // [RING][16] (L_kk, ~ 1 / L_kk) of the staged diagonal tiles
  unsigned long long * bars;
  long long *sdoff, *sooff;
  int *rec, *alist, *iscr;
  signed char * st;
  // per problem
  const double *base, *a, *C, *bl, *bu, *xl, *xu;
  double *Rg, *Qg;
  int q, nrec;
  long long qoff;
  double f;
  TriWarp tw; // the serial warp: the structured solves
  int sw; // the warp that runs the serial parts (solves, Givens records, R solve): rotated over the CTAs of an SM, whose
          // warps 0 would otherwise all sit on the same scheduler while the three others idle

  static __host__ __device__ long long ring_doubles(int nb) { return TriWarp::ring_doubles(nb); }

  __device__ BlockGi(const BlockGiParams & p, double * sm)
  : P(p), n(p.G.n), mc(p.mc), m(p.mc + p.nb), T(blockDim.x), tid(threadIdx.x), lane(threadIdx.x & 31), warp(threadIdx.x >> 5),
    W(blockDim.x >> 5), up(p.G.type == SG_ARROW_UP)
  {
    const int ne = (n + 2) & ~1;
    x = sm;
    z = x + ne;
    d = z + ne;
    w = d + ne;
    u = w + ne;
    r = u + ne;
    scr = r + ne;
    hred = scr + 80; // 2 x 128 class sums of a Householder application (double-buffered) + the scaled dot
    rtri = hred + 264; // blocked R solve: RB x (R_kk, ~ 1 / R_kk, R_{k-1,k}, -)
    MJ = (n + 127) / 128;
    qring = rtri + 4 * RB; // [QD][MJ][128]
    rtau = qring + QD * MJ * 128; // tau of record e (0 for a Givens record)
    Lt = rtau + ((p.max_iter + 1) & ~1);
    Bt = Lt + p.G.nmax * p.G.nmax;
    ring = Bt + p.G.nmax * p.G.nmax + ((2 * p.G.nmax * p.G.nmax) & 1); // 16-byte aligned (bulk copies)
    dgp = reinterpret_cast<double2 *>(ring + (p.fast_nb ? ring_doubles(p.fast_nb) - RING * 32 : 0));
    bars = reinterpret_cast<unsigned long long *>(ring + ring_doubles(p.fast_nb));
    sdoff = reinterpret_cast<long long *>(bars + (p.fast_nb ? RING : 0));
    sooff = sdoff + (p.fast_nb ? p.G.b : 0);
    rec = reinterpret_cast<int *>(sooff + (p.fast_nb ? p.G.b : 0));
    alist = rec + 3 * p.max_iter;
    iscr = alist + n;
    st = reinterpret_cast<signed char *>(iscr + 16);
    double * slot = p.ws + (long long)blockIdx.x * p.ws_stride;
    Rg = slot;
    Qg = slot + (long long)n * (n + 1) / 2;
    unsigned nsm;
    asm("mov.u32 %0, %%nsmid;" : "=r"(nsm));
    sw = (int)((blockIdx.x / max(1u, nsm)) % (unsigned)(blockDim.x >> 5));
    tw.ring = ring;
    tw.dgp = dgp;
    tw.bars = bars;
    tw.sdoff = sdoff;
    tw.sooff = sooff;
    tw.base = nullptr;
    tw.b = p.G.b;
    tw.n = n;
    tw.lane = lane;
    tw.rph = 0u;
  }

  static __host__ __device__ long long smem_bytes(int n, int nmax, int m, int max_iter, int fast_nb, int b)
  {
    const long long ne = (n + 2) & ~1;
    const long long tiles = 2LL * nmax * nmax + ((2LL * nmax * nmax) & 1);
    const long long fast = fast_nb ? ring_doubles(fast_nb) + RING + 2LL * b : 0;
    const long long qst = (long long)QD * ((n + 127) / 128) * 128 + ((max_iter + 1) & ~1);
    return (6 * ne + 80 + 264 + 4 * RB + qst + tiles + fast) * 8 + (3LL * max_iter + n + 16) * 4 + ((m + 15) & ~15);
  }

  // once per kernel: barriers of the ring, block offsets of G in shared memory (the solves read them on their critical path)
  __device__ void setup()
  {
    if(P.fast_nb)
    {
      if(tid == 0) tw.init_barriers();
      for(int i = tid; i < P.G.b; i += T)
      {
        sdoff[i] = P.G.doff[i];
        sooff[i] = i + 1 < P.G.b ? P.G.ooff[i] : 0;
      }
    }
    __syncthreads();
  }

  __device__ __forceinline__ int pidx(int i) const { return up ? sg_perm(P.G, i) : i; }
  __device__ __forceinline__ static long long colR(int k) { return (long long)k * (k + 1) / 2; }

  // C.col(p).dot(v) (StructuredC::col + SingleNZSegmentVector::dot): dot4 over the rows of the block
  __device__ __forceinline__ double col_dot(int p, const double * v) const
  {
    const int bi = P.toblock[p];
    const double * c = C + P.coff[bi] + (long long)(p - P.ccstr0[bi]) * P.cld[bi];
    return dot4_rows(P.cnvar[bi], c, 1, v + P.cvar0[bi], 1);
  }

  // dot32(len, a, b) by warp 0, result to every thread. a, b: global or shared.
  __device__ __forceinline__ double block_dot32(int len, const double * pa, const double * pb)
  {
    __syncthreads();
    if(warp == 0)
    {
      double acc = 0;
      for(int k = lane; k < len; k += 32) acc = fma(pa[k], pb[k], acc);
      for(int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(BG_FULL, acc, off);
      if(lane == 0) scr[0] = acc;
    }
    __syncthreads();
    return scr[0];
  }

  // lexicographic minimum of (val, idx) over the CTA; threads without a candidate pass idx = INT_MAX
  __device__ __forceinline__ void block_first_min(double & val, int & idx)
  {
    for(int off = 16; off >= 1; off >>= 1)
    {
      const double ov = __shfl_xor_sync(BG_FULL, val, off);
      const int oi = __shfl_xor_sync(BG_FULL, idx, off);
      if(oi != 0x7fffffff && (idx == 0x7fffffff || ov < val || (ov == val && oi < idx)))
      {
        val = ov;
        idx = oi;
      }
    }
    if(W > 1)
    {
      __syncthreads();
      if(lane == 0)
      {
        scr[8 + warp] = val;
        iscr[warp] = idx;
      }
      __syncthreads();
      val = scr[8];
      idx = iscr[0];
      for(int k = 1; k < W; ++k)
      {
        const double ov = scr[8 + k];
        const int oi = iscr[k];
        if(oi != 0x7fffffff && (idx == 0x7fffffff || ov < val || (ov == val && oi < idx)))
        {
          val = ov;
          idx = oi;
        }
      }
    }
  }

  // ---- OrthonormalSequence::applyTransposeToTheLeft / applyToTheLeft on a vector in shared memory.
  // One Householder record = a reflector of up to n entries stored in the CTA's global slice (L2): applied by the WHOLE
  // CTA. The inner product E.w runs over 128 classes (k mod 128, ascending k in each: thread t owns the classes t, t + T,
  // ...), which are folded (c, c+32), (c+64, c+96) and then reduced by the dot32 butterfly — the order the oracle
  // defines (oracle/block_oracle.hpp); every entry of the reflector is loaded once, all loads of a record in flight
  // together. Round 1 applied a record with one warp: 12 dependent L2 round trips per pass at n = 384, two passes per
  // record, ~100 records, twice per iteration — 95 % of a solve (profiles/r01zc_blockgi_E_tri.json: 4.8 k QP/s).
  static constexpr int MAXE = ME; // entries of a reflector per thread: 128 classes x ME >= n (n <= 512: 4, n <= 1024: 8)

  // entries k = tid, tid + 128, ... of the reflector of record e (1.0 for the implicit leading entry), and its tau:
  // loaded one record AHEAD of their use, so that the L2 / HBM latency of a record hides behind the reduction of the
  // previous one (the record list of a config-E solve does not fit L2: ncu, profiles/r02y_*: L2 hit rate 21 %, the dot
  // of the reflector 19 % of the stall samples, all long_scoreboard)
  __device__ __forceinline__ void load_reflector(int e, double (&pk)[MAXE], double & tau) const
  {
    const int start = rec[3 * e], size = rec[3 * e + 1];
    const double * p = Qg + rec[3 * e + 2];
    tau = 0.0;
#pragma unroll
    for(int j = 0; j < MAXE; ++j) pk[j] = 0.0;
    if(start >= 0)
    {
      tau = p[0];
      if(tid < 128)
      {
#pragma unroll
        for(int j = 0; j < MAXE; ++j)
        {
          const int k = tid + 128 * j;
          if(k < size) pk[j] = k == 0 ? 1.0 : p[k];
        }
      }
    }
  }

  // H = I - tau E E^T applied to v(0:len), E held in registers (load_reflector). The inner product E.w runs over 128
  // classes (k mod 128, ascending k in each), folded (c, c+32), (c+64, c+96) and reduced by the dot32 butterfly: the order
  // the oracle defines (oracle/block_oracle.hpp).
  __device__ __forceinline__ void householder(const double (&pk)[MAXE], double tau, int len, double * v)
  {
    if(tid < 128)
    {
      double acc = 0.0;
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = tid + 128 * j;
        if(k < len) acc = fma(pk[j], v[k], acc);
      }
      hred[tid] = acc;
    }
    __syncthreads();
    if(warp == 0)
    {
      double acc = (hred[lane] + hred[lane + 32]) + (hred[lane + 64] + hred[lane + 96]);
      for(int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(BG_FULL, acc, off);
      if(lane == 0) hred[256] = tau * acc;
    }
    __syncthreads();
    const double hd = hred[256];
    if(tid < 128)
    {
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = tid + 128 * j;
        if(k < len) v[k] = fma(-hd, pk[j], v[k]);
      }
    }
    __syncthreads();
  }

  // one Givens record (c[size], s[size] at p) applied by warp 0 to vs[0 .. size] in shared memory
  __device__ __forceinline__ void givens_record(double * vs, const double * p, const int size, const int dir)
  {
    if(dir > 0)
    {
      // Givens(c, s)^T, i ascending: x' = c x - s y, y' = s x + c y; the y' of one rotation is the x of the next
      double carry = vs[0];
      for(int i0 = 0; i0 < size; i0 += 32)
      {
        const int k = min(i0 + lane, size - 1);
        const double cl = p[k], sl = p[size + k];
        const int cn = min(32, size - i0);
#pragma unroll 4
        for(int j = 0; j < cn; ++j)
        {
          const double c = __shfl_sync(BG_FULL, cl, j), sn = __shfl_sync(BG_FULL, sl, j);
          const double xi = carry, yi = vs[i0 + j + 1];
          const double nx = fma(c, xi, -(sn * yi));
          carry = fma(c, yi, sn * xi);
          if(lane == 0) vs[i0 + j] = nx;
        }
      }
      if(lane == 0) vs[size] = carry;
    }
    else
    {
      // Givens(c, s), i descending: x' = c x + s y, y' = -s x + c y; the x' of one rotation is the y of the next
      double carry = vs[size];
      for(int i1 = size; i1 > 0; i1 -= 32)
      {
        const int cn = min(32, i1);
        const int k = max(i1 - 1 - lane, 0);
        const double cl = p[k], sl = p[size + k];
#pragma unroll 4
        for(int j = 0; j < cn; ++j)
        {
          const int i = i1 - 1 - j;
          const double c = __shfl_sync(BG_FULL, cl, j), sn = __shfl_sync(BG_FULL, sl, j);
          const double xi = vs[i], yi = carry;
          carry = fma(c, xi, sn * yi);
          const double ny = fma(c, yi, -(sn * xi));
          if(lane == 0) vs[i + 1] = ny;
        }
      }
      if(lane == 0) vs[0] = carry;
    }
  }

  // the same with c (cs[0 .. size)) and s (cs[soff .. soff + size)) staged in shared memory: uniform loads, no shuffle
  __device__ __forceinline__ void givens_record_staged(double * vs, const double * cs, const int soff, const int size, const int dir)
  {
    if(dir > 0)
    {
      double carry = vs[0];
#pragma unroll 4
      for(int i = 0; i < size; ++i)
      {
        const double c = cs[i], sn = cs[soff + i];
        const double xi = carry, yi = vs[i + 1];
        const double nx = fma(c, xi, -(sn * yi));
        carry = fma(c, yi, sn * xi);
        if(lane == 0) vs[i] = nx;
      }
      if(lane == 0) vs[size] = carry;
    }
    else
    {
      double carry = vs[size];
#pragma unroll 4
      for(int i = size - 1; i >= 0; --i)
      {
        const double c = cs[i], sn = cs[soff + i];
        const double xi = vs[i], yi = carry;
        carry = fma(c, xi, sn * yi);
        const double ny = fma(c, yi, -(sn * xi));
        if(lane == 0) vs[i + 1] = ny;
      }
      if(lane == 0) vs[0] = carry;
    }
  }

  // dir = +1: Q^T v (records in order of addition), dir = -1: Q v (reverse order)
  __device__ void apply_sequence_smem(double * v, const int dir)
  {
    if(nrec > 0)
    {
      double pc[MAXE], pn[MAXE], tc, tn = 0.0;
      int e = dir > 0 ? 0 : nrec - 1;
      load_reflector(e, pc, tc);
      for(int cnt = 0; cnt < nrec; ++cnt, e += dir)
      {
        const int en = e + dir;
        if(cnt + 1 < nrec) load_reflector(en, pn, tn);
        const int start = rec[3 * e], size = rec[3 * e + 1];
        double * vs = v + (start & 0x7fffffff);
        if(start >= 0)
          householder(pc, tc, size, vs);
        else
        {
          if(warp == 0) givens_record(vs, Qg + rec[3 * e + 2], size, dir);
          __syncthreads();
        }
#pragma unroll
        for(int j = 0; j < MAXE; ++j) pc[j] = pn[j];
        tc = tn;
      }
    }
    __syncthreads();
  }

  // The reflector of record e travels to the thread that uses it as cp.async copies into a thread-PRIVATE slot of a
  // QD-deep stage (entry k of v belongs to thread k mod 128, so the thread that issues a copy is the only one that ever
  // reads it: no barrier, no register held while the copy is in flight); entries outside [start, end) are not copied.
  // One commit group per call (empty for a Givens record or past the end), so that wait_group<QD - 1> always means "the
  // record about to be applied has landed".
  __device__ __forceinline__ void issue_record(const int e, const bool valid, const int kt) const
  {
    if(valid)
    {
      const int s = rec[3 * e], en = s + rec[3 * e + 1];
      if(s < 0 && warp == sw)
      {
        // a Givens record: c and s of its rotations, when they fit the slot (they are read by warp 0 after a barrier)
        const int sz = rec[3 * e + 1];
        if(sz <= MJ * 64)
        {
          const double * p = Qg + rec[3 * e + 2];
          double * slot = qring + ((unsigned)e % QD) * MJ * 128;
          for(int k = lane; k < sz; k += 32)
          {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(bg_smem_addr(slot + k)), "l"(p + k) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(bg_smem_addr(slot + MJ * 64 + k)), "l"(p + sz + k) : "memory");
          }
        }
      }
      if(s >= 0 && tid < 128)
      {
        const double * p = Qg + rec[3 * e + 2];
        double * slot = qring + ((unsigned)e % QD) * MJ * 128 + tid;
#pragma unroll
        for(int j = 0; j < MAXE; ++j)
        {
          if(j < MJ)
          {
            const int k = kt + 128 * j;
            if(k >= s && k < en) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(bg_smem_addr(slot + 128 * j)), "l"(p + (k - s)) : "memory");
          }
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }

  // pk[j] = E[tid + 128 j - start] inside [start, end), 1.0 for the implicit leading entry, 0 elsewhere; st: start (sign
  // bit: a Givens record), en: one past the end
  __device__ __forceinline__ void take_record(const int e, const int kt, double (&pk)[MAXE], double & tau, int & st, int & en) const
  {
    const int s = rec[3 * e], sz = rec[3 * e + 1];
    st = s;
    en = (s & 0x7fffffff) + sz;
    tau = rtau[e];
    asm volatile("cp.async.wait_group %0;" ::"n"(QD - 1) : "memory");
    const double * slot = qring + ((unsigned)e % QD) * MJ * 128 + (tid & 127);
#pragma unroll
    for(int j = 0; j < MAXE; ++j)
    {
      const int k = kt + 128 * j;
      const double t = (j < MJ && k > s && k < en) ? slot[128 * j] : 0.0; // (entries outside the record were not copied)
      pk[j] = k == s ? 1.0 : t;
    }
  }

  __device__ __forceinline__ void prefetch_record_l2(const int e) const
  {
    const int len = rec[3 * e] >= 0 ? rec[3 * e + 1] : 2 * rec[3 * e + 1];
    const double * p = Qg + rec[3 * e + 2];
    if(8 * tid < len) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + 8 * tid)); // one request per 64 bytes (128 threads: 1024 doubles >= n)
    if(8 * tid + 1024 < len) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + 8 * tid + 1024)); // (a Givens record of n > 512)
  }

  // one record applied to the register-resident vector (see apply_sequence_reg)
  __device__ __forceinline__ void apply_record(const int e, const int dir, const int kt, double * v, double (&vr)[MAXE], const double (&pc)[MAXE],
                                               const double tc, const int st, const int en, int & buf)
  {
    if(st >= 0)
    {
      double * h = hred + 128 * buf;
      double acc = 0.0;
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        const double t = fma(pc[j], vr[j], acc);
        acc = (k >= st && k < en) ? t : acc;
      }
      if(tid < 128) h[(tid - st) & 127] = acc;
      __syncthreads();
      double a4 = (h[lane] + h[lane + 32]) + (h[lane + 64] + h[lane + 96]);
#pragma unroll
      for(int off = 16; off >= 1; off >>= 1) a4 += __shfl_xor_sync(BG_FULL, a4, off);
      const double hd = tc * a4;
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        const double t = fma(-hd, pc[j], vr[j]);
        vr[j] = (k >= st && k < en) ? t : vr[j];
      }
      buf ^= 1;
    }
    else
    {
      // a Givens sequence is a serial chain over adjacent entries: through shared memory, on warp 0
      const int s0 = st & 0x7fffffff; // rotations on the entries s0 .. en (en = s0 + number of rotations)
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        if(k >= s0 && k <= en) v[k] = vr[j];
      }
      __syncthreads();
      if(warp == sw)
      {
        if(en - s0 <= MJ * 64)
          givens_record_staged(v + s0, qring + ((unsigned)e % QD) * MJ * 128, MJ * 64, en - s0, dir);
        else
          givens_record(v + s0, Qg + rec[3 * e + 2], en - s0, dir);
      }
      __syncthreads();
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        if(k >= s0 && k <= en) vr[j] = v[k];
      }
    }
  }

  // ---- the same sequence with the vector in REGISTERS (round 2). Thread t (< 128) owns v[t], v[t + 128], ... for the
  // whole pass, so a reflector needs ONE barrier (the 128 class sums through shared memory; every warp then folds and
  // reduces them redundantly, no second barrier to hand the result back) instead of three, and nothing of v moves
  // between records. The classes of the inner product are those of the oracle: entry k of a reflector that starts at
  // `start` belongs to class k mod 128, i.e. to the thread that owns v[start + k] — thread t runs class (t - start) mod
  // 128, ascending k in it: the same chains, folds and butterfly, the same bits. The next record is fetched into a second
  // register set while the current one is applied (two sets used alternately: no copies), records further down the list
  // are pulled into L2 (the list of a config-E solve, ~ 0.4 MB per CTA, does not stay there: profiles/r02y_*).
  __device__ void apply_sequence_reg(double * v, const int dir)
  {
    constexpr int PFD = 8; // records of look-ahead of the L2 prefetch
    if(nrec > 0)
    {
      const int kt = tid < 128 ? tid : 0x40000000; // (threads beyond the 128 classes own nothing)
      double vr[MAXE];
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        vr[j] = k < n ? v[k] : 0.0;
      }
      double pc[MAXE], tc;
      int sc, ec;
      int e = dir > 0 ? 0 : nrec - 1;
      for(int a = 1; a < PFD && a < nrec; ++a) prefetch_record_l2(e + dir * a);
      for(int a = 0; a < QD - 1; ++a) issue_record(e + dir * a, a < nrec, kt);
      int buf = 0;
#pragma unroll 1
      for(int left = nrec; left > 0; --left, e += dir)
      {
        if(left > PFD) prefetch_record_l2(e + dir * PFD);
        issue_record(e + dir * (QD - 1), left > QD - 1, kt);
        take_record(e, kt, pc, tc, sc, ec);
        apply_record(e, dir, kt, v, vr, pc, tc, sc, ec, buf);
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
      for(int j = 0; j < MAXE; ++j)
      {
        const int k = kt + 128 * j;
        if(k < n) v[k] = vr[j];
      }
    }
    __syncthreads();
  }

  __device__ void apply_sequence(double * v, const int dir)
  {
    if(P.flags & BGF_REG_SEQUENCE)
      apply_sequence_reg(v, dir);
    else
      apply_sequence_smem(v, dir);
  }
  __device__ void apply_qt(double * v) { apply_sequence(v, +1); }
  __device__ void apply_q(double * v) { apply_sequence(v, -1); }

  // StructuredG::solveL / solveInPlaceLTranspose on v (shared memory), every thread of the CTA; ends on a barrier
  __device__ void g_solve(double * v, const bool transpose, const int start, const int end)
  {
    if(P.fast_nb && (P.flags & BGF_WARP_SOLVE))
    {
      if(warp == sw)
      {
        TriWarp t = tw; // (a local copy: its address, not the solver's, is what the out-of-line exact path sees)
        t.base = base;
        if(P.fast_nb == 8)
        {
          if(transpose)
            t.solve<8, true>(v, start, end);
          else
            t.solve<8, false>(v, start, end);
        }
        else if(P.fast_nb == 12)
        {
          if(transpose)
            t.solve<12, true>(v, start, end);
          else
            t.solve<12, false>(v, start, end);
        }
        else
        {
          if(transpose)
            t.solve<16, true>(v, start, end);
          else
            t.solve<16, false>(v, start, end);
        }
        tw.rph = t.rph;
      }
      __syncthreads();
    }
    else
      sg_solve_inplace(P.G, base, v, Lt, Bt, transpose, start, end);
  }

  // ---- r = R^-1 d1 (StructuredQR::RSolve), blocked by RB columns: the triangle of a block sits in the registers of warp 0
  // (lane j: row k0 + j; every load of the block in flight at once, ONE L2 round trip per RB links instead of one per
  // link), the substitution inside it is the uniform-pivot recurrence with proven quotients, and the rows above the block
  // take the block's RB updates from all the threads (descending k for every entry: the order of the column-oriented
  // loop, same bits). On entry w(0:q) = d(0:q), visible to every thread.
  __device__ void r_solve_blocked()
  {
    for(int k1 = q; k1 > 0; k1 -= RB)
    {
      const int k0 = max(0, k1 - RB), nbk = k1 - k0;
      if(warp == sw)
      {
        const int lc = min(lane, nbk - 1);
        const double w0 = w[k0 + lc];
        bool done;
        {
          // column k0 + c of the triangle in Tc[c] (row k0 + lane; rows below the diagonal read the diagonal). A partial
          // block (the last one: nbk < RB) runs the same straight-line code with its missing links switched off.
          double Tc[RB];
#pragma unroll
          for(int c = 0; c < RB; ++c)
          {
            const int cc = min(c, nbk - 1);
            Tc[c] = Rg[colR(k0 + cc) + k0 + min(lc, cc)];
          }
          // link c reads (R_cc, ~ 1 / R_cc, R_{c-1,c}): written by lane c from two loads of its own (no register indexed by the lane)
          const double dg = Rg[colR(k0 + lc) + k0 + lc];
          const double sup = Rg[colR(k0 + lc) + k0 + max(lc - 1, 0)];
          if(lane < RB) reinterpret_cast<double4 *>(rtri)[lane] = make_double4(dg, bg_rcp(dg), sup, 0.0);
          const double4 * tri = reinterpret_cast<const double4 *>(rtri);
          __syncwarp();
          double wj = w0;
          double wp = __shfl_sync(BG_FULL, wj, nbk - 1);
#pragma unroll
          for(int c = RB - 1; c >= 0; --c)
          {
            const bool act = c < nbk; // (uniform)
            const double tn = __shfl_sync(BG_FULL, wj, c > 0 ? c - 1 : 0);
            const double4 t4 = tri[c];
            const double q0 = wp * t4.y;
            const double e = fma(-t4.x, q0, wp);
            const double rk = fma(e, t4.y, q0);
            if(c > 0)
            {
              const double wn = fma(-rk, t4.z, tn);
              wp = act ? wn : wp;
            }
            if(act && lane < c) wj = fma(-rk, Tc[c], wj); // (a lane stops at its own link: it is left holding its pivot)
          }
          // lane c: its own quotient again (same operands, same bits) and the proof that it is correctly rounded
          const double4 own = tri[min(lane, RB - 1)];
          const double q0 = wj * own.y;
          const double eo = fma(-own.x, q0, wj);
          const double rv = fma(eo, own.y, q0);
          const bool ok = lane >= nbk || div_proof(wj, own.x, rv);
          done = __all_sync(BG_FULL, ok);
          if(done && lane < nbk) r[k0 + lane] = rv;
          __syncwarp();
        }
        if(!done)
        {
          // an unproven quotient (rare): one link at a time, true divisions
          JRLQP_FB_HIT_IF(lane == 0, FB_R_SOLVE);
          double wj = w0, rv = 0.0;
          const double dg = Rg[colR(k0 + lc) + k0 + lc];
#pragma unroll 1
          for(int c = nbk - 1; c >= 0; --c)
          {
            const double rk = __shfl_sync(BG_FULL, wj, c) / __shfl_sync(BG_FULL, dg, c);
            const double tc = Rg[colR(k0 + c) + k0 + min(lc, c)];
            rv = lane == c ? rk : rv;
            const double nw = fma(-rk, tc, wj);
            wj = lane < c ? nw : wj;
          }
          if(lane < nbk) r[k0 + lane] = rv;
        }
      }
      __syncthreads();
      for(int j = tid; j < k0; j += T)
      {
        double wv = w[j];
#pragma unroll
        for(int c = RB - 1; c >= 0; --c)
          if(c < nbk) wv = fma(-r[k0 + c], Rg[colR(k0 + c) + j], wv);
        w[j] = wv;
      }
      __syncthreads();
    }
  }

  // ---- selectViolatedConstraint_ (src/experimental/BlockGISolver.cpp:111-164)
  __device__ __forceinline__ void slacks(int i, double & sl, double & su) const
  {
    if(i < mc)
    {
      const double cx = col_dot(i, x);
      sl = cx - bl[i];
      su = bu[i] - cx;
    }
    else
    {
      const int j = i - mc;
      sl = x[j] - xl[j];
      su = xu[j] - x[j];
    }
  }

  // returns the constraint index (-1: none) and its status
  __device__ int select(int & status)
  {
    double best = 0.0;
    int code = 0x7fffffff;
    bool both = false;
    for(int i = tid; i < m; i += T)
    {
      if(st[i] != BG_INACTIVE) continue;
      double sl, su;
      slacks(i, sl, su);
      const bool nl = sl < 0.0, nu = su < 0.0;
      both |= nl && nu;
      const double v = nl ? sl : su;
      const int ci = 2 * i + (nl ? 0 : 1);
      if((nl || nu) && (code == 0x7fffffff || v < best)) // i ascending inside a thread: strict < keeps the first
      {
        best = v;
        code = ci;
      }
    }
    if(__syncthreads_or(both))
    {
      // bl > bu somewhere: the `else if` chain of the reference is order dependent, replay it literally
      if(tid == 0)
      {
        double smin = 0;
        int c = 0x7fffffff;
        for(int i = 0; i < m; ++i)
        {
          if(st[i] != BG_INACTIVE) continue;
          double sl, su;
          slacks(i, sl, su);
          if(sl < smin)
          {
            smin = sl;
            c = 2 * i;
          }
          else if(su < smin)
          {
            smin = su;
            c = 2 * i + 1;
          }
        }
        iscr[8] = c;
      }
      __syncthreads();
      code = iscr[8];
      __syncthreads();
    }
    else
      block_first_min(best, code);
    if(code == 0x7fffffff)
    {
      status = BG_INACTIVE;
      return -1;
    }
    const int p = code >> 1;
    status = p < mc ? ((code & 1) ? BG_UPPER : BG_LOWER) : ((code & 1) ? BG_UPPER_BOUND : BG_LOWER_BOUND);
    return p;
  }

  // ---- computeStep_ (src/experimental/BlockGISolver.cpp:166-174)
  __device__ void compute_step(int p, int status)
  {
    // d = Q^T L^-1 n+ (StructuredJ::premultByJt)
    for(int i = tid; i < n; i += T) w[i] = 0.0;
    __syncthreads();
    int hs, he;
    if(status <= BG_EQUALITY)
    {
      const int bi = P.toblock[p];
      const int rows = P.cnvar[bi], s0 = P.cvar0[bi];
      const double * c = C + P.coff[bi] + (long long)(p - P.ccstr0[bi]) * P.cld[bi];
      for(int i = tid; i < rows; i += T) w[pidx(s0 + i)] = c[i];
      hs = s0;
      he = s0 + rows;
    }
    else
    {
      const int b = p - mc;
      if(tid == 0) w[pidx(b)] = status == BG_UPPER_BOUND ? -1.0 : 1.0;
      hs = b;
      he = b + 1;
    }
    __syncthreads();
    g_solve(w, false, hs, he);
    const bool neg = status == BG_UPPER;
    for(int i = tid; i < n; i += T) d[i] = neg ? -w[i] : w[i];
    __syncthreads();
    apply_qt(d);
    // z = L^-T Q [0; d2] (StructuredJ::premultByJ2)
    for(int i = tid; i < n; i += T) w[i] = i < q ? 0.0 : d[i];
    __syncthreads();
    apply_q(w);
    g_solve(w, true, 0, -1);
    for(int i = tid; i < n; i += T) z[i] = w[pidx(i)];
    __syncthreads();
    // r = R^-1 d1 (StructuredQR::RSolve): column-oriented back substitution, true division
    for(int k = tid; k < q; k += T) w[k] = d[k];
    __syncthreads();
    if(P.flags & BGF_BLOCKED_RSOLVE)
    {
      r_solve_blocked();
      return;
    }
    for(int k = q - 1; k >= 0; --k)
    {
      const double * Rk = Rg + colR(k);
      const double rk = w[k] / Rk[k];
      if(tid == 0) r[k] = rk;
      for(int j = tid; j < k; j += T) w[j] = fma(-rk, Rk[j], w[j]);
      __syncthreads();
    }
  }

  // ---- StructuredQR::add (src/structured/StructuredQR.cpp:72-86); false: the record storage is full
  __device__ bool add_constraint(int p, int status)
  {
    const int len = n - q;
    if(nrec >= P.max_iter || qoff + len > P.qcap) return false;
    const double c0 = d[q];
    const double tailSq = len == 1 ? 0.0 : block_dot32(len - 1, d + q + 1, d + q + 1);
    double * pe = Qg + qoff;
    double tau, beta;
    if(tailSq <= 2.2250738585072014e-308) // (std::numeric_limits<double>::min)()
    {
      tau = 0.0;
      beta = c0;
      for(int i = 1 + tid; i < len; i += T) pe[i] = 0.0;
    }
    else
    {
      beta = sqrt(fma(c0, c0, tailSq));
      if(c0 >= 0.0) beta = -beta;
      const double den = c0 - beta;
      for(int i = 1 + tid; i < len; i += T) pe[i] = d[q + i] / den;
      tau = (beta - c0) / beta;
    }
    double * Rq = Rg + colR(q);
    for(int k = tid; k < q; k += T) Rq[k] = d[k];
    if(tid == 0)
    {
      pe[0] = tau;
      Rq[q] = beta;
      rtau[nrec] = tau;
      rec[3 * nrec] = q;
      rec[3 * nrec + 1] = len;
      rec[3 * nrec + 2] = (int)qoff;
      st[p] = (signed char)status; // DualSolver::addConstraint: A_.activate
      alist[q] = p;
    }
    qoff += len;
    ++nrec;
    ++q;
    __syncthreads();
    return true;
  }

  // ---- DualSolver::removeConstraint + StructuredQR::remove (src/DualSolver.cpp:237-244, StructuredQR.cpp:88-103)
  __device__ bool remove_constraint(int l)
  {
    // u.segment(l, q - l) = u.tail(q - l) (u has q + 1 entries); A_.deactivate(l)
    const int qa = q;
    __syncthreads();
    for(int k0 = l; k0 < qa; k0 += T)
    {
      const int k = k0 + tid;
      const double un = k < qa ? u[k + 1] : 0.0;
      const int an = k + 1 < qa ? alist[k + 1] : -1;
      const int gone = alist[l];
      __syncthreads();
      if(k0 == l && tid == 0) st[gone] = BG_INACTIVE;
      if(k < qa)
      {
        u[k] = un;
        if(k + 1 < qa) alist[k] = an;
      }
      __syncthreads();
    }
    --q;
    const int g = q - l;
    if(g <= 0) return true; // the last constraint: an empty Givens sequence
    if(nrec >= P.max_iter || qoff + 2 * g > P.qcap) return false;
    double * cs = Qg + qoff;
    for(int i = l; i < q; ++i)
    {
      double * Ri = Rg + colR(i);
      const double * Ri1 = Rg + colR(i + 1);
      for(int k = tid; k < i; k += T) Ri[k] = Ri1[k];
      double c, s, rr;
      bg_make_givens(Ri1[i], Ri1[i + 1], c, s, rr);
      __syncthreads(); // everybody has read R(i, i+1), R(i+1, i+1)
      if(tid == 0)
      {
        Ri[i] = rr;
        cs[i - l] = c;
        cs[g + i - l] = s;
      }
      for(int j = i + 2 + tid; j <= q; j += T) // rows i, i+1 of the columns to the right, rotated by Qi^T
      {
        double * Rj = Rg + colR(j);
        const double xi = Rj[i], yi = Rj[i + 1];
        Rj[i] = fma(c, xi, -(s * yi));
        Rj[i + 1] = fma(c, yi, s * xi);
      }
      __syncthreads();
    }
    if(tid == 0)
    {
      rtau[nrec] = 0.0;
      rec[3 * nrec] = l | (int)0x80000000;
      rec[3 * nrec + 1] = g;
      rec[3 * nrec + 2] = (int)qoff;
    }
    qoff += 2 * g;
    ++nrec;
    __syncthreads();
    return true;
  }

  __device__ void write_failure(long long b, int status)
  {
    for(int i = tid; i < n; i += T) P.x[b * n + i] = 0.0;
    if(P.u)
      for(int i = tid; i < m; i += T) P.u[b * m + i] = 0.0;
    if(P.act)
      for(int i = tid; i < m; i += T) P.act[b * m + i] = 0;
    if(P.alist)
      for(int i = tid; i < n; i += T) P.alist[b * n + i] = -1;
    if(tid == 0)
    {
      if(P.f) P.f[b] = 0.0;
      if(P.iters) P.iters[b] = 0;
      if(P.status) P.status[b] = status;
      if(P.nact) P.nact[b] = 0;
      if(P.qdoubles) P.qdoubles[b] = 0;
    }
  }

  __device__ void write_result(long long b, int status, int it)
  {
    __syncthreads();
    for(int i = tid; i < n; i += T) P.x[b * n + i] = x[i];
    if(P.u)
    {
      // DualSolver::multipliers (src/DualSolver.cpp:38-69)
      for(int i = tid; i < m; i += T) P.u[b * m + i] = 0.0;
      __syncthreads();
      for(int k = tid; k < q; k += T)
      {
        const int i = alist[k];
        const int s = st[i];
        P.u[b * m + i] = (s == BG_UPPER || s == BG_UPPER_BOUND) ? u[k] : -u[k];
      }
    }
    if(P.act)
      for(int i = tid; i < m; i += T) P.act[b * m + i] = st[i];
    if(P.alist)
      for(int i = tid; i < n; i += T) P.alist[b * n + i] = i < q ? alist[i] : -1;
    if(tid == 0)
    {
      if(P.f) P.f[b] = f;
      if(P.iters) P.iters[b] = it;
      if(P.status) P.status[b] = status;
      if(P.nact) P.nact[b] = q;
      if(P.qdoubles) P.qdoubles[b] = qoff;
    }
  }

  __device__ void solve(long long b)
  {
    base = P.G.data + b * P.G.stride;
    a = P.a + b * P.sa;
    C = P.C + b * P.sC;
    bl = P.bl + b * P.sbl;
    bu = P.bu + b * P.sbu;
    xl = P.nb ? P.xl + b * P.sxl : nullptr;
    xu = P.nb ? P.xu + b * P.sxu : nullptr;
    q = 0;
    nrec = 0;
    qoff = 0;
    __syncthreads();

    // processInitialActiveSet (src/experimental/BlockGISolver.cpp:293-377), cold start: equalities of the data
    // would be activated here, and initializePrimalDualPoints asserts there is none (:474)
    int neq = 0;
    for(int i = tid; i < m; i += T)
    {
      st[i] = BG_INACTIVE;
      neq += i < mc ? (bl[i] == bu[i]) : (xl[i - mc] == xu[i - mc]);
    }
    neq = __syncthreads_count(neq) ? 1 : 0; // (a count of threads; only zero / non-zero and > n matter below)
    if(neq)
    {
      // exact count for the OVERCONSTRAINED test
      int cnt = 0;
      if(tid == 0)
      {
        for(int i = 0; i < m; ++i) cnt += i < mc ? (bl[i] == bu[i]) : (xl[i - mc] == xu[i - mc]);
        iscr[8] = cnt;
      }
      __syncthreads();
      cnt = iscr[8];
      __syncthreads();
      write_failure(b, cnt > n ? 6 /* OVERCONSTRAINED_PROBLEM */ : 1 /* INCONSISTENT_INPUT */);
      return;
    }
    if(!P.llt_ok[b * P.ok_stride])
    {
      write_failure(b, 2 /* NON_POS_HESSIAN */);
      return;
    }
    // initializePrimalDualPoints (:476-481): x = -G^-1 a, f = 0.5 a.x
    for(int i = tid; i < n; i += T) w[pidx(i)] = a[i];
    __syncthreads();
    g_solve(w, false, 0, -1);
    g_solve(w, true, 0, -1);
    for(int i = tid; i < n; i += T) x[i] = -w[pidx(i)];
    f = 0.5 * block_dot32(n, a, x);

    // DualSolver::solve (src/DualSolver.cpp:96-168)
    bool skip1 = false;
    int p = -1, status = BG_INACTIVE;
    int it = 0;
    for(; it < P.max_iter; ++it)
    {
      if(!skip1)
      {
        p = select(status);
        if(status == BG_INACTIVE)
        {
          write_result(b, 0, it);
          return;
        }
        if(tid == 0) u[q] = 0.0;
      }
      compute_step(p, status);

      // computeStepLength_ (src/experimental/BlockGISolver.cpp:176-243)
      double t1 = P.big_bnd;
      int l = 0x7fffffff;
      for(int k = tid; k < q; k += T)
      {
        const int sk = st[k]; // the reference indexes the status by the POSITION k (:188), kept
        if(sk != BG_EQUALITY && sk != BG_FIXED && r[k] > 0.0)
        {
          const double tk = u[k] / r[k];
          if(tk < t1)
          {
            t1 = tk;
            l = k;
          }
        }
      }
      block_first_min(t1, l);
      if(l == 0x7fffffff)
      {
        t1 = P.big_bnd;
        l = 0;
      }
      const double znorm = sqrt(block_dot32(n, z, z));
      double t2 = P.big_bnd, ndot = 0.0;
      if(znorm > 1e-14)
      {
        double bnd, cx, cz;
        if(status <= BG_EQUALITY)
        {
          __syncthreads();
          if(tid == 0) scr[2] = col_dot(p, x);
          if(tid == T - 1) scr[3] = col_dot(p, z);
          __syncthreads();
          cx = scr[2];
          cz = scr[3];
          bnd = status == BG_LOWER ? bl[p] : bu[p];
          ndot = status == BG_UPPER ? -cz : cz;
        }
        else
        {
          const int pb = p - mc;
          cx = x[pb];
          cz = z[pb];
          bnd = status == BG_LOWER_BOUND ? xl[pb] : xu[pb];
          ndot = status == BG_UPPER_BOUND ? -cz : cz;
        }
        t2 = (bnd - cx) / cz;
      }
      const double t = t2 < t1 ? t2 : t1; // std::min(t1, t2)
      if(t >= P.big_bnd)
      {
        write_result(b, 3 /* INFEASIBLE */, it);
        return;
      }
      __syncthreads();
      if(t2 >= P.big_bnd)
      {
        for(int k = tid; k < q; k += T) u[k] = fma(-t, r[k], u[k]);
        if(tid == 0) u[q] += t;
        if(!remove_constraint(l))
        {
          write_result(b, 7 /* UNKNOWN: record storage exhausted */, it);
          return;
        }
        skip1 = true;
      }
      else
      {
        for(int i = tid; i < n; i += T) x[i] = fma(t, z[i], x[i]);
        f += (t * ndot) * (0.5 * t + u[q]);
        __syncthreads(); // u[q] read by everybody before it changes
        for(int k = tid; k < q; k += T) u[k] = fma(-t, r[k], u[k]);
        if(tid == 0) u[q] += t;
        bool ok;
        if(t == t2)
        {
          ok = add_constraint(p, status);
          skip1 = false;
        }
        else
        {
          ok = remove_constraint(l);
          skip1 = true;
        }
        if(!ok)
        {
          write_result(b, 7, it);
          return;
        }
      }
    }
    write_result(b, 4 /* MAX_ITER_REACHED */, it);
  }
};

// compiled for 4 resident CTAs per SM (register cap 65536 / (128 * 4); measured: profiles/r4d_*)
template<int ME>
__global__ void __launch_bounds__(128, 4) blockgi_kernel(const BlockGiParams P)
{
  extern __shared__ __align__(16) double sm[];
  __shared__ long long next;
  BlockGi<ME> S(P, sm);
  S.setup();
  for(;;)
  {
    __syncthreads();
    if(threadIdx.x == 0) next = (long long)atomicAdd(P.ticket, 1ULL);
    __syncthreads();
    const long long b = next;
    if(b >= P.batch) break;
    S.solve(b);
  }
}

// Test harness (tests/test_orthonormal_sequence.py; tests/InternalTest.cpp:35-323 of the reference): the solver's OWN
// apply_q / apply_qt run on a record list given by the caller — records in the layout add_constraint / remove_constraint
// write (rec = (start | sign bit for Givens, size, offset), data in the Q slice of the workspace) — on `ncases` vectors.
__global__ void blockgi_sequence_test_kernel(const BlockGiParams P, const int * rec_in, int nrec, double * v, int ncases, int transpose)
{
  extern __shared__ __align__(16) double sm[];
  BlockGi<8> S(P, sm);
  for(int i = threadIdx.x; i < 3 * nrec; i += blockDim.x) S.rec[i] = rec_in[i];
  for(int i = threadIdx.x; i < nrec; i += blockDim.x) S.rtau[i] = rec_in[3 * i] >= 0 ? S.Qg[rec_in[3 * i + 2]] : 0.0;
  S.nrec = nrec;
  for(int cs = blockIdx.x; cs < ncases; cs += gridDim.x)
  {
    __syncthreads();
    for(int i = threadIdx.x; i < S.n; i += blockDim.x) S.w[i] = v[(long long)cs * S.n + i];
    __syncthreads();
    if(transpose)
      S.apply_qt(S.w);
    else
      S.apply_q(S.w);
    for(int i = threadIdx.x; i < S.n; i += blockDim.x) v[(long long)cs * S.n + i] = S.w[i];
  }
}

} // namespace jrlqp
