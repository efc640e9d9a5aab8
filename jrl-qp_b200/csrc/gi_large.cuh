// Dense Goldfarb-Idnani solver for LARGE problems (128 < n <= 1024): one QP per CTA of T threads,
// persistent work-queue kernel, sm_100a. Same reference path as gi_dense_cta.cuh
//   GoldfarbIdnaniSolver::solve -> DualSolver::solve -> {init_, selectViolatedConstraint_,
//   computeStep_, computeStepLength_, addConstraint_, removeConstraint_}
//   (src/GoldfarbIdnaniSolver.cpp:18-338, src/DualSolver.cpp:38-244, src/internal/ActiveSet.cpp)
// and the same canonical arithmetic (oracle/gi_oracle.cpp): results are bit-identical to the oracle
// and to the shared-memory kernel. What differs is where the per-QP state lives: an n x n matrix no
// longer fits in shared memory (MultiIK fixtures of the reference, tests/MultiIK.zip: n = 387 and
// n = 210; 1.2 MB for one J), so every CTA owns a workspace in global memory — re-used from problem
// to problem by the persistent CTA, hence resident in the 126 MB L2 — and only the vectors, the
// status / active-list arrays and the rotation table stay in shared memory.
//
// Workspace of one CTA (doubles):
//   Lw  n x ldl column-major: lower triangle of G -> L in place. Column-major makes the two O(n^3)
//       loops coalesced: thread = row i reads L(i, j) (consecutive i), L(k, j) comes from a staged
//       copy of row k in shared memory (Cholesky) / from a uniform vector load (J build).
//   Jr  n x ldl row-major: J = L^-T is BUILT here with thread = column j (J(k, j), consecutive j).
//   Jc  = Lw's storage, column-major: J is transposed into it once L is no longer needed (32 x 32
//       tiles through shared memory). The main loop wants rows across the lanes: z = J2 d2 and the
//       column rotations of add / drop read and write J(i, c) for consecutive i => coalesced.
//       d = J^T n+ walks columns (thread = column j, 32-byte vector loads: every sector fetched is used).
//   Rp  packed upper-triangular R, column k at k (k + 1) / 2.
//   Bw  (warm start only) n x ldl column-major: B = L^-1 N, then its Householder QR in place.
#pragma once

#include "gi_dense_cta.cuh"

namespace jrlqp
{

constexpr int kRingStages = 3; // stages of the TMA-fed column ring (see GiLarge::ring_*)

// Shared-memory carve-up, computed identically on the host (size) and on the device (pointers).
struct LargeSmem
{
  int nv; // padded vector length (multiple of 4)
  int off_x, off_z, off_d, off_r, off_u, off_cv, off_gc, off_gs, off_gcs, off_ldiag, off_rinv, off_w, off_rowk, off_scr, off_redd, off_tile;
  int off_bact, off_hco, off_alp;
  int off_alist, off_gk, off_iscr, off_redi, off_stat, off_eq;
  int total; // doubles
  __host__ __device__ LargeSmem(int n, int m, bool warm)
  {
    nv = (n + 3) & ~3;
    int o = 0;
    off_x = o, o += nv;
    off_z = o, o += nv;
    off_d = o, o += nv;
    off_r = o, o += nv;
    off_u = o, o += nv + 4;
    off_cv = o, o += nv;
    off_gc = o, o += nv;
    off_gs = o, o += nv;
    off_gcs = o, o += 2 * nv;
    off_ldiag = o, o += nv;
    off_rinv = o, o += nv;
    off_w = o, o += nv;
    off_rowk = o, o += nv;
    off_scr = o, o += 32;
    off_redd = o, o += 64;
    off_tile = o, o += 32 * 33 + 1;
    o += o & 1;
    off_bact = off_hco = off_alp = o;
    if(warm)
    {
      off_bact = o, o += nv;
      off_hco = o, o += nv;
      off_alp = o, o += nv;
    }
    off_alist = o, o += nv / 2 + 2;
    off_gk = o, o += nv / 2 + 2;
    off_iscr = o, o += 8;
    off_redi = o, o += 32;
    off_stat = o, o += (m + 7) / 8 + 1;
    off_eq = o, o += (m + 7) / 8 + 1;
    total = o;
  }
};

// shared memory behind the LargeSmem carve-up (doubles): the column ring with its barriers, then the slab of the warm start
__host__ __device__ inline long long large_ring_doubles(int n, int ring_cols)
{
  const long long ldl = (n + 3) & ~3;
  return ring_cols > 0 ? (long long)kRingStages * ring_cols * ldl + ((kRingStages + 1) & ~1) : 0;
}
__host__ __device__ inline long long large_slab_doubles(int n, int slab_rows)
{
  return slab_rows > 0 ? (long long)n * slab_rows + 2ll * ((n + 1) & ~1) + 16 : 0;
}

__host__ __device__ inline long long large_workspace_doubles(int n, bool warm)
{
  const long long ldl = (n + 3) & ~3;
  long long w = 2ll * n * ldl + ((long long)n * (n + 1) / 2 + 3) / 4 * 4;
  if(warm) w += (long long)n * ldl;
  return w;
}

template<int T, bool WARM>
struct GiLarge
{
  static constexpr int NW = T / 32;
  static constexpr int CH = 16; // values in flight per thread in the constraint scan
  static constexpr int PF = 4; // rotations per chunk when the Givens table is applied
  static constexpr int RP = 1024 / T; // rows per thread at the largest supported n
  const GiParams & P;
  const int tid, lane, warp;
  const int n, mc, nb, m, ldl;
  // global workspace of this CTA
  double *Lw, *Jr, *Jc, *Rp, *Bw;
  // shared memory
  double *xs, *zs, *ds, *rs, *us, *cv, *gc, *gs, *ldiag, *rinv, *wv, *rowk, *scr, *redd, *tile, *bact, *hco, *alp;
  double2 * gcs;
  int *alist, *gk, *iscr, *redi;
  signed char *stat, *eqf;
  // TMA-fed column ring (rcols > 0): kRingStages stages of rcols consecutive columns of the column-major J, filled by
  // cp.async.bulk copies that complete on one mbarrier per stage; rph holds the phase bit of every stage (uniform)
  double * ring;
  unsigned long long * rbar;
  int rcols;
  unsigned rph;
  // warm start: slab of srows rows of J (all columns) for J = J Q, two buffers for the essential part of a reflector, tau tmp per row
  double * slab;
  int srows;
  // per-problem views
  const double *Cb, *bl, *bu, *xl, *xu;
  long long ldC;
  bool cvec;
  // solver state (uniform)
  int q;
  double f;

  __device__ GiLarge(const GiParams & p, double * smem, double * work)
  : P(p), tid(threadIdx.x), lane(threadIdx.x & 31), warp(threadIdx.x >> 5), n(p.n), mc(p.mc), nb(p.nb), m(p.mc + p.nb), ldl((p.n + 3) & ~3)
  {
    const LargeSmem S(n, m, WARM);
    xs = smem + S.off_x;
    zs = smem + S.off_z;
    ds = smem + S.off_d;
    rs = smem + S.off_r;
    us = smem + S.off_u;
    cv = smem + S.off_cv;
    gc = smem + S.off_gc;
    gs = smem + S.off_gs;
    gcs = reinterpret_cast<double2 *>(smem + S.off_gcs);
    ldiag = smem + S.off_ldiag;
    rinv = smem + S.off_rinv;
    wv = smem + S.off_w;
    rowk = smem + S.off_rowk;
    scr = smem + S.off_scr;
    redd = smem + S.off_redd;
    tile = smem + S.off_tile;
    bact = smem + S.off_bact;
    hco = smem + S.off_hco;
    alp = smem + S.off_alp;
    alist = reinterpret_cast<int *>(smem + S.off_alist);
    gk = reinterpret_cast<int *>(smem + S.off_gk);
    iscr = reinterpret_cast<int *>(smem + S.off_iscr);
    redi = reinterpret_cast<int *>(smem + S.off_redi);
    stat = reinterpret_cast<signed char *>(smem + S.off_stat);
    eqf = reinterpret_cast<signed char *>(smem + S.off_eq);
    Lw = work;
    Jc = work;
    Jr = work + (long long)n * ldl;
    Rp = work + 2ll * n * ldl;
    Bw = Rp + ((long long)n * (n + 1) / 2 + 3) / 4 * 4;
    rcols = p.ring_cols;
    ring = smem + ((S.total + 1) & ~1);
    rbar = reinterpret_cast<unsigned long long *>(ring + (long long)kRingStages * rcols * ldl);
    rph = 0u;
    slab = ring + large_ring_doubles(n, rcols);
    srows = p.slab_rows;
  }

  // ------------------------------------------------------------------------------------------
  // Column ring. The rotation sweep of an add and z = J2 d2 stream J column by column (3 KB per column at n = 387) out of a
  // per-CTA workspace that lives in L2 / HBM: with plain loads a thread has PF = 4 values in flight and the phases are bound
  // by the memory latency (profiles/r5h_*: long_scoreboard 55 % of the samples, issue slots 16 % busy). Here ONE thread asks
  // the TMA unit for the next chunks of rcols whole columns (contiguous in the column-major storage: one bulk copy per
  // chunk), two chunks ahead of the chunk being used; the threads read their rows from shared memory. Protocol per chunk:
  // wait on the stage's mbarrier (phase bit in rph) -> use -> block barrier -> the stage is refilled. Writes of J stay plain
  // global stores; a pass starts with fence.proxy.async.global + block barrier so that the bulk copies (async proxy) see them.
  // ------------------------------------------------------------------------------------------
  __device__ __forceinline__ static unsigned saddr(const void * p) { return (unsigned)__cvta_generic_to_shared(p); }
  __device__ void ring_setup()
  {
    if(rcols > 0 && tid == 0)
    {
      for(int i = 0; i < kRingStages; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(saddr(rbar + i)));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  // (one thread) columns [c0, c0 + nc) of J -> stage
  __device__ __forceinline__ void ring_issue(const int stage, const int c0, const int nc)
  {
    const unsigned bar = saddr(rbar + stage);
    const unsigned bytes = (unsigned)(nc * ldl * 8);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // earlier generic reads of this stage are done (block barrier)
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(saddr(ring + (long long)stage * rcols * ldl)),
                 "l"(Jc + (long long)c0 * ldl), "r"(bytes), "r"(bar)
                 : "memory");
  }
  __device__ __forceinline__ void ring_wait(const int stage)
  {
    const unsigned bar = saddr(rbar + stage), par = (rph >> stage) & 1u;
    unsigned done;
    do
    {
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(done) : "r"(bar), "r"(par) : "memory");
    } while(!done);
    rph ^= 1u << stage;
  }
  // chunk k of a DESCENDING pass that starts at column n - 1: columns [max(0, hi - rcols + 1), hi], hi = n - 1 - k rcols
  __device__ __forceinline__ void ring_issue_down(const int k)
  {
    const int hi = n - 1 - k * rcols, st = max(0, hi - rcols + 1);
    ring_issue(k % kRingStages, st, hi - st + 1);
  }
  // chunk k of an ASCENDING pass that starts at column c0: columns [c0 + k rcols, min(n, c0 + (k + 1) rcols))
  __device__ __forceinline__ void ring_issue_up(const int c0, const int k)
  {
    const int st = c0 + k * rcols;
    ring_issue(k % kRingStages, st, min(rcols, n - st));
  }

  // the rotation sweep of add_constraint() through the ring: rows tid and tid + T of J (n <= 2 T), links n - 2 ... lo
  __device__ void add_rotations_ring(const int lo)
  {
    const int r0 = tid, r1 = tid + T;
    const bool h0 = r0 < n, h1 = r1 < n;
    asm volatile("fence.proxy.async.global;" ::: "memory");
    sync();
    const int nch = (n - lo + rcols - 1) / rcols;
    if(tid == 0)
      for(int k = 0; k < kRingStages - 1 && k < nch; ++k) ring_issue_down(k);
    double y0 = 0.0, y1 = 0.0;
#pragma unroll 1
    for(int k = 0; k < nch; ++k)
    {
      if(tid == 0 && k + kRingStages - 1 < nch) ring_issue_down(k + kRingStages - 1);
      const int hi = n - 1 - k * rcols, st = max(0, hi - rcols + 1);
      ring_wait(k % kRingStages);
      const double * sb = ring + (long long)(k % kRingStages) * rcols * ldl - (long long)st * ldl; // sb[c * ldl + row] = J(row, c)
      int i = hi;
      if(k == 0)
      {
        y0 = h0 ? sb[(long long)(n - 1) * ldl + r0] : 0.0;
        y1 = h1 ? sb[(long long)(n - 1) * ldl + r1] : 0.0;
        i = n - 2;
      }
      const int ilo = max(st, lo);
#pragma unroll 4
      for(; i >= ilo; --i)
      {
        const double2 cs2 = gcs[i];
        const double c = cs2.x, sn = cs2.y;
        const double * col = sb + (long long)i * ldl;
        double * out = Jc + (long long)(i + 1) * ldl;
        if(h0)
        {
          const double xi = col[r0];
          out[r0] = fma(c, y0, sn * xi);
          y0 = fma(c, xi, -(sn * y0));
        }
        if(h1)
        {
          const double xi = col[r1];
          out[r1] = fma(c, y1, sn * xi);
          y1 = fma(c, xi, -(sn * y1));
        }
      }
      if(k + 1 < nch) sync(); // every thread is done with this stage before it is refilled
    }
    if(h0) Jc[(long long)lo * ldl + r0] = y0;
    if(h1) Jc[(long long)lo * ldl + r1] = y1;
  }

  // z = J2 d2 through the ring (rows tid and tid + T): the first chunks were requested by compute_step() before d was formed
  __device__ void z_ring()
  {
    const int r0 = tid, r1 = tid + T;
    const bool h0 = r0 < n, h1 = r1 < n;
    const int nch = (n - q + rcols - 1) / rcols;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, b0 = 0, b1 = 0, b2 = 0, b3 = 0;
#pragma unroll 1
    for(int k = 0; k < nch; ++k)
    {
      if(tid == 0 && k + kRingStages - 1 < nch) ring_issue_up(q, k + kRingStages - 1);
      const int st = q + k * rcols, en = min(n, st + rcols);
      ring_wait(k % kRingStages);
      const double * sb = ring + (long long)(k % kRingStages) * rcols * ldl - (long long)st * ldl;
      const double * p0 = sb + (h0 ? r0 : 0);
      const double * p1 = sb + (h1 ? r1 : 0);
      int c = st;
#pragma unroll 2
      for(; c + 3 < en; c += 4)
      {
        const double d0 = ds[c], d1 = ds[c + 1], d2 = ds[c + 2], d3 = ds[c + 3];
        a0 = fma(p0[(long long)c * ldl], d0, a0);
        a1 = fma(p0[(long long)(c + 1) * ldl], d1, a1);
        a2 = fma(p0[(long long)(c + 2) * ldl], d2, a2);
        a3 = fma(p0[(long long)(c + 3) * ldl], d3, a3);
        b0 = fma(p1[(long long)c * ldl], d0, b0);
        b1 = fma(p1[(long long)(c + 1) * ldl], d1, b1);
        b2 = fma(p1[(long long)(c + 2) * ldl], d2, b2);
        b3 = fma(p1[(long long)(c + 3) * ldl], d3, b3);
      }
      // (only the last chunk has a tail: the chunks before it hold a multiple of four columns)
      if(c < en)
      {
        a0 = fma(p0[(long long)c * ldl], ds[c], a0);
        b0 = fma(p1[(long long)c * ldl], ds[c], b0);
      }
      if(c + 1 < en)
      {
        a1 = fma(p0[(long long)(c + 1) * ldl], ds[c + 1], a1);
        b1 = fma(p1[(long long)(c + 1) * ldl], ds[c + 1], b1);
      }
      if(c + 2 < en)
      {
        a2 = fma(p0[(long long)(c + 2) * ldl], ds[c + 2], a2);
        b2 = fma(p1[(long long)(c + 2) * ldl], ds[c + 2], b2);
      }
      if(k + 1 < nch) sync();
    }
    if(h0) zs[r0] = (a0 + a1) + (a2 + a3);
    if(h1) zs[r1] = (b0 + b1) + (b2 + b3);
  }

  __device__ __forceinline__ static long long colR(int k) { return ((long long)k * (k + 1)) >> 1; }
  __device__ __forceinline__ void sync() const { __syncthreads(); }

  // ------------------------------------------------------------------------------------------
  // Cholesky of G in the column-major workspace Lw (Eigen llt_inplace, src/GoldfarbIdnaniSolver.cpp:58-61)
  // Canonical order: left-looking, v_i = G(i,k) - dot4_{j<k}(L(i,j), L(k,j)). Returns false when a
  // pivot is not positive (NON_POS_HESSIAN).
  // ------------------------------------------------------------------------------------------
  __device__ bool cholesky(long long b)
  {
    const double * __restrict__ Gb = P.G + b * P.sG;
    const int ldg = P.ldg;
    // stage the lower triangle (column-major in HBM and in the workspace: coalesced both ways)
    for(int j = 0; j < n; ++j)
      for(int i = j + tid; i < n; i += T) Lw[i + (long long)j * ldl] = __ldg(Gb + i + (long long)j * ldg);
    sync();
#pragma unroll 1
    for(int k = 0; k < n; ++k)
    {
      // row k of L (strided in the column-major storage) staged once for all the threads
      for(int j = tid; j < k; j += T) rowk[j] = Lw[k + (long long)j * ldl];
      sync();
      double v[RP];
#pragma unroll
      for(int s = 0; s < RP; ++s)
      {
        const int i = k + tid + s * T;
        v[s] = 0.0;
        if(i < n)
        {
          const double * Li = Lw + i;
          double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
          int j = 0;
#pragma unroll 2
          for(; j + 3 < k; j += 4)
          {
            const double l0 = Li[(long long)j * ldl], l1 = Li[(long long)(j + 1) * ldl], l2 = Li[(long long)(j + 2) * ldl],
                         l3 = Li[(long long)(j + 3) * ldl];
            a0 = fma(l0, rowk[j], a0);
            a1 = fma(l1, rowk[j + 1], a1);
            a2 = fma(l2, rowk[j + 2], a2);
            a3 = fma(l3, rowk[j + 3], a3);
          }
          if(j < k) a0 = fma(Li[(long long)j * ldl], rowk[j], a0);
          if(j + 1 < k) a1 = fma(Li[(long long)(j + 1) * ldl], rowk[j + 1], a1);
          if(j + 2 < k) a2 = fma(Li[(long long)(j + 2) * ldl], rowk[j + 2], a2);
          v[s] = Li[(long long)k * ldl] - ((a0 + a1) + (a2 + a3));
          if(i == k) scr[0] = v[s];
        }
      }
      sync();
      const double vk = scr[0];
      if(vk <= 0.0) return false; // Eigen llt: "if (x <= 0) return k" (uniform)
      const double lkk = sqrt(vk);
#pragma unroll
      for(int s = 0; s < RP; ++s)
      {
        const int i = k + tid + s * T;
        if(i == k)
        {
          Lw[k + (long long)k * ldl] = lkk;
          ldiag[k] = lkk;
          rinv[k] = 1.0 / lkk;
        }
        else if(i < n)
          Lw[i + (long long)k * ldl] = v[s] / lkk;
      }
      sync();
    }
    // optional copy-out of L (what the reference leaves in G)
    if(P.L != nullptr)
    {
      double * Lout = P.L + b * (long long)n * n;
      for(int j = 0; j < n; ++j)
        for(int i = j + tid; i < n; i += T) Lout[i + (long long)j * n] = Lw[i + (long long)j * ldl];
    }
    return true;
  }

  // x = -G^-1 a by ONE warp (column-oriented forward / backward substitution, true division), f = a.x / 2
  __device__ void initial_point(const double * __restrict__ ab, const double * __restrict__ Lw)
  {
    for(int i = lane; i < n; i += 32) wv[i] = __ldg(ab + i);
    __syncwarp();
#pragma unroll 1
    for(int k = 0; k < n; ++k)
    {
      const double yk = wv[k] / ldiag[k];
      const double * Lk = Lw + (long long)k * ldl;
      __syncwarp();
      if(lane == 0) wv[k] = yk;
      for(int i = k + 1 + lane; i < n; i += 32) wv[i] = fma(-yk, Lk[i], wv[i]);
      __syncwarp();
    }
#pragma unroll 1
    for(int k = n - 1; k >= 0; --k)
    {
      const double xk = wv[k] / ldiag[k];
      __syncwarp();
      if(lane == 0) wv[k] = xk;
      for(int i = lane; i < k; i += 32) wv[i] = fma(-xk, Lw[k + (long long)i * ldl], wv[i]);
      __syncwarp();
    }
    double facc = 0.0;
    for(int i = lane; i < n; i += 32)
    {
      const double xi = -wv[i];
      xs[i] = xi;
      facc = fma(__ldg(ab + i), xi, facc); // dot32: lane = k & 31, ascending k
    }
    const double fs = 0.5 * warp_sum32(facc);
    if(lane == 0) scr[1] = fs;
  }

  // x = -G^-1 a and f = a.x / 2 by the WHOLE CTA (used when the factor is shared by the batch and no other work can
  // hide a serial warp): the two triangular solves run over 32-row diagonal blocks. The block itself is a serial
  // chain on warp 0 (rows over the lanes, the block of L in the shared-memory tile, quotients from the stored
  // reciprocals with their proof of correct rounding); the rows outside it are then updated by all the threads
  // (one row per thread, 32 independent coalesced loads). Every element still receives its updates
  // w_i = fma(-y_k, L(i,k), w_i) in ascending k (forward) / fma(-x_k, L(k,i), w_i) in descending k (backward), with a
  // true division by the diagonal: the same operations as initial_point(), bit for bit.
  __device__ void initial_point_blocked(const double * __restrict__ ab, const double * __restrict__ L)
  {
    for(int i = tid; i < n; i += T) wv[i] = __ldg(ab + i);
    sync();
    const int nblk = (n + 31) >> 5;
#pragma unroll 1
    for(int pass = 0; pass < 2; ++pass)
    {
#pragma unroll 1
      for(int bi = 0; bi < nblk; ++bi)
      {
        const int r0 = 32 * (pass == 0 ? bi : nblk - 1 - bi);
        const int nb = min(32, n - r0);
        if(warp == 0)
        {
          // tile[jj * 33 + lane] = L(r0 + lane, r0 + jj), lower part of the diagonal block (coalesced along the rows)
          const double * Lb = L + r0 + (long long)r0 * ldl;
#pragma unroll 8
          for(int jj = 0; jj < nb; ++jj) tile[jj * 33 + lane] = (lane < nb && lane >= jj) ? Lb[lane + (long long)jj * ldl] : 0.0;
          __syncwarp();
          const int rl = min(r0 + lane, n - 1);
          double w = wv[rl];
          const double ld = ldiag[rl], ri = rinv[rl];
          if(pass == 0)
          {
#pragma unroll 1
            for(int jj = 0; jj < nb; ++jj)
            {
              bool ok;
              double cand = div_rcp(w, ld, ri, ok);
              if(!ok && lane == jj) cand = w / ld; // only the lane whose entry is final matters
              JRLQP_FB_HIT_IF(!ok && lane == jj, FB_LARGE_INIT);
              const double yk = __shfl_sync(JRLQP_FULL, cand, jj);
              if(lane == jj)
                w = yk;
              else if(lane > jj)
                w = fma(-yk, tile[jj * 33 + lane], w);
            }
          }
          else
          {
#pragma unroll 1
            for(int jj = nb - 1; jj >= 0; --jj)
            {
              bool ok;
              double cand = div_rcp(w, ld, ri, ok);
              if(!ok && lane == jj) cand = w / ld; // only the lane whose entry is final matters
              JRLQP_FB_HIT_IF(!ok && lane == jj, FB_LARGE_INIT);
              const double xk = __shfl_sync(JRLQP_FULL, cand, jj);
              if(lane == jj)
                w = xk;
              else if(lane < jj)
                w = fma(-xk, tile[lane * 33 + jj], w); // L(r0 + jj, r0 + lane)
            }
          }
          if(lane < nb) wv[r0 + lane] = w;
        }
        sync();
        if(pass == 0)
        {
          // rows below the block: w_i -= sum_k y_k L(i, k), k ascending over the block
          for(int i = r0 + nb + tid; i < n; i += T)
          {
            const double * Li = L + i + (long long)r0 * ldl;
            double acc = wv[i];
#pragma unroll 1
            for(int j0 = 0; j0 < nb; j0 += 8)
            {
              double lv[8];
#pragma unroll
              for(int u = 0; u < 8; ++u) lv[u] = j0 + u < nb ? Li[(long long)(j0 + u) * ldl] : 0.0;
#pragma unroll
              for(int u = 0; u < 8; ++u)
                if(j0 + u < nb) acc = fma(-wv[r0 + j0 + u], lv[u], acc);
            }
            wv[i] = acc;
          }
        }
        else
        {
          // rows above the block: w_i -= sum_k x_k L(k, i), k descending over the block (32 contiguous entries of column i)
          for(int i = tid; i < r0; i += T)
          {
            const double * Lc = L + r0 + (long long)i * ldl;
            double acc = wv[i];
#pragma unroll 1
            for(int j0 = ((nb - 1) & ~7); j0 >= 0; j0 -= 8)
            {
              double lv[8];
#pragma unroll
              for(int u = 0; u < 8; ++u) lv[u] = j0 + u < nb ? Lc[j0 + u] : 0.0;
#pragma unroll
              for(int u = 7; u >= 0; --u)
                if(j0 + u < nb) acc = fma(-wv[r0 + j0 + u], lv[u], acc);
            }
            wv[i] = acc;
          }
        }
        sync();
      }
    }
    if(warp == 0)
    {
      double facc = 0.0;
      for(int i = lane; i < n; i += 32)
      {
        const double xi = -wv[i];
        xs[i] = xi;
        facc = fma(__ldg(ab + i), xi, facc); // dot32: lane = k & 31, ascending k
      }
      const double fs = 0.5 * warp_sum32(facc);
      if(lane == 0) scr[1] = fs;
    }
  }

  // J = L^-T built row-major in Jr (upper triangle only; the strict lower triangle is never read),
  // thread = column j, by the warps [w0, NW): J(i,j) = (-dot4_{k=i+1..j}(L(k,i), J(k,j))) * (1 / L(i,i))
  __device__ void build_J(int w0)
  {
    const int nwb = NW - w0;
    if(warp < w0) return;
    for(int j0 = 32 * (warp - w0); j0 < n; j0 += 32 * nwb)
    {
      const int j = j0 + lane;
      const int jc = min(j, n - 1);
      const int jmax = min(n - 1, j0 + 31);
      if(j < n) Jr[(long long)j * ldl + j] = rinv[j];
      __syncwarp();
#pragma unroll 1
      for(int r = jmax - 1; r >= 0; --r)
      {
        double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        const double * Lr = Lw + (long long)r * ldl; // column r of L: L(k, r), uniform across the lanes
        // columns j < k0 of this warp have no entry in row k0: their accumulations are discarded
        const int kstart = r + 1;
#pragma unroll 1
        for(int k0 = kstart; k0 <= jmax; k0 += 4)
        {
          const double * Jk = Jr + (long long)k0 * ldl + jc;
          const bool v1 = k0 + 1 <= jmax, v2 = k0 + 2 <= jmax, v3 = k0 + 3 <= jmax;
          const double l0 = Lr[k0];
          const double l1 = v1 ? Lr[k0 + 1] : 0.0;
          const double l2 = v2 ? Lr[k0 + 2] : 0.0;
          const double l3 = v3 ? Lr[k0 + 3] : 0.0;
          const double j0v = k0 <= j ? Jk[0] : 0.0;
          const double j1v = (v1 && k0 + 1 <= j) ? Jk[ldl] : 0.0;
          const double j2v = (v2 && k0 + 2 <= j) ? Jk[2 * (long long)ldl] : 0.0;
          const double j3v = (v3 && k0 + 3 <= j) ? Jk[3 * (long long)ldl] : 0.0;
          const double t0 = fma(l0, j0v, a0);
          const double t1 = fma(l1, j1v, a1);
          const double t2 = fma(l2, j2v, a2);
          const double t3 = fma(l3, j3v, a3);
          a0 = k0 <= j ? t0 : a0;
          a1 = k0 + 1 <= j ? t1 : a1;
          a2 = k0 + 2 <= j ? t2 : a2;
          a3 = k0 + 3 <= j ? t3 : a3;
        }
        if(r < j && j < n) Jr[(long long)r * ldl + j] = (-((a0 + a1) + (a2 + a3))) * rinv[r];
        // a column only depends on L and on itself (same lane): no synchronisation needed
      }
    }
  }

  // Jc(i, j) = i <= j ? Jr(i, j) : 0, column-major, 32 x 32 tiles through shared memory (whole CTA)
  __device__ void transpose_J()
  {
    const int nt = (n + 31) / 32;
    for(int t = 0; t < nt * nt; ++t)
    {
      const int ti = t / nt, tj = t % nt; // tile rows 32 ti.., columns 32 tj..
      sync();
      for(int e = tid; e < 1024; e += T)
      {
        const int r = e >> 5, c = e & 31; // coalesced along the columns of the row-major source
        const int i = 32 * ti + r, j = 32 * tj + c;
        tile[r * 33 + c] = (i < n && j < n && i <= j) ? Jr[(long long)i * ldl + j] : 0.0;
      }
      sync();
      for(int e = tid; e < 1024; e += T)
      {
        const int c = e >> 5, r = e & 31; // coalesced along the rows of the column-major destination
        const int i = 32 * ti + r, j = 32 * tj + c;
        if(i < n && j < n) Jc[i + (long long)j * ldl] = tile[r * 33 + c];
      }
    }
    sync();
  }

  // ---- factor shared by the batch (P.pre, see gi_params.h)
  __device__ __forceinline__ const double * pre_L() const { return P.pre + 2ll * n * ldl; }
  // diag(L), 1 / diag(L) into shared memory, optional copy-out of L. False: G is not positive definite.
  __device__ bool load_prefactor(long long b)
  {
    if(*P.pre_ok == 0) return false;
    const int nv = (n + 3) & ~3;
    const double * pd = P.pre + 3ll * n * ldl;
    for(int i = tid; i < n; i += T)
    {
      ldiag[i] = pd[i];
      rinv[i] = pd[nv + i];
    }
    if(P.L != nullptr)
    {
      const double * Lk = pre_L();
      double * Lout = P.L + b * (long long)n * n;
      for(int j = 0; j < n; ++j)
        for(int i = j + tid; i < n; i += T) Lout[i + (long long)j * n] = Lk[i + (long long)j * ldl];
    }
    sync();
    return true;
  }
  // Jc <- shared J (column-major, n x ldl), by the warps [w0, NW), 16-byte vectors
  __device__ void copy_pre_J(int w0)
  {
    if(warp < w0) return;
    const long long total2 = ((long long)n * ldl) >> 1; // ldl is a multiple of 4
    const double2 * src = reinterpret_cast<const double2 *>(P.pre);
    double2 * dst = reinterpret_cast<double2 *>(Jc);
    const int nth = T - 32 * w0, t = tid - 32 * w0;
#pragma unroll 8
    for(long long e = t; e < total2; e += nth) dst[e] = __ldg(src + e);
  }

  // init_ (src/GoldfarbIdnaniSolver.cpp:56-82)
  __device__ bool init(long long b)
  {
    const double * __restrict__ ab = P.a + b * P.sa;
    if(mc > 0 && P.sC != 0)
    {
      // pull this problem's C towards L2 while the factorisation runs (shared C is resident anyway)
      const char * Cg = reinterpret_cast<const char *>(P.C + b * P.sC);
      const long long bytes = ((long long)(mc - 1) * P.ldc + n) * 8;
      for(long long o = (long long)tid * 128; o < bytes; o += (long long)T * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(Cg + o));
    }
    if(P.pre != nullptr)
    {
      // G is shared by the batch: its factor was computed once for the launch (gi_large_prefactor_kernel, same code,
      // same bits). The CTA copies J = L^-T, then computes x = -G^-1 a from the shared L.
      if(!load_prefactor(b)) return false;
      copy_pre_J(0);
      initial_point_blocked(ab, pre_L());
      sync();
      f = scr[1];
    }
    else
    {
      if(!cholesky(b)) return false;
      // warp 0: x = -G^-1 a (serial division chain) while the other warps build J
      if(warp == 0) initial_point(ab, Lw);
      build_J(1);
      sync();
      f = scr[1];
      transpose_J(); // L is no longer needed: J moves into its storage, column-major
    }
    for(int c = tid; c < m; c += T)
    {
      stat[c] = ST_INACTIVE; // A_.reset()
      eqf[c] = (c < mc ? (bl[c] == bu[c]) : (xl[c - mc] == xu[c - mc])) ? 1 : 0; // initActiveSet's tests, once
    }
    q = 0;
    sync();
    return true;
  }

  // ------------------------------------------------------------------------------------------
  // selectViolatedConstraint_ (src/GoldfarbIdnaniSolver.cpp:84-134), thread = constraint
  // ------------------------------------------------------------------------------------------
  __device__ Sel select()
  {
    double best = 0.0;
    int code = JRLQP_NONE;
    bool bothneg = false;
    for(int base = 0; base < mc; base += T)
    {
      const int c = base + tid;
      const bool act = c < mc && stat[c] == ST_INACTIVE;
      if(__ballot_sync(JRLQP_FULL, act) == 0u) continue; // warp-uniform
      const double * ci = Cb + (long long)min(c, mc - 1) * ldC;
      const double blc = act ? bl[c] : 0.0, buc = act ? bu[c] : 0.0;
      // C shared by the batch: scan its transposed copy (made once per call, coalesced across the constraints);
      // lanes whose constraint is active issue no memory request
      const double cx = P.ct != nullptr ? dot4_col<CH, true>(P.ct + ct_offset(min(c, mc - 1), n), xs, n, act)
                                        : (cvec ? dot4_row<true, CH>(ci, xs, n, act) : dot4_row<false, CH>(ci, xs, n, act));
      if(act)
      {
        const double sl = cx - blc;
        const double su = buc - cx;
        if(sl < 0.0 && su < 0.0) bothneg = true;
        if(sl < best)
        {
          best = sl;
          code = c * 8 + ST_LOWER;
        }
        else if(su < best)
        {
          best = su;
          code = c * 8 + ST_UPPER;
        }
      }
    }
    for(int base = 0; base < nb; base += T)
    {
      const int c = base + tid;
      if(c < nb && stat[mc + c] == ST_INACTIVE)
      {
        const double xi = xs[c];
        const double sl = xi - xl[c];
        const double su = xu[c] - xi;
        if(sl < 0.0 && su < 0.0) bothneg = true;
        if(sl < best)
        {
          best = sl;
          code = (mc + c) * 8 + ST_LOWER_BOUND;
        }
        else if(su < best)
        {
          best = su;
          code = (mc + c) * 8 + ST_UPPER_BOUND;
        }
      }
    }
    // first-minimum reduction: smallest value, ties to the smallest constraint index. (A thread sees
    // its own constraints in ascending order with a strict test, so its candidate is its first minimum.)
#pragma unroll
    for(int off = 16; off >= 1; off >>= 1)
    {
      const double ov = __shfl_xor_sync(JRLQP_FULL, best, off);
      const int oc = __shfl_xor_sync(JRLQP_FULL, code, off);
      if(ov < best || (ov == best && oc < code))
      {
        best = ov;
        code = oc;
      }
    }
    const unsigned anyneg_w = __ballot_sync(JRLQP_FULL, bothneg);
    if(lane == 0)
    {
      redd[warp] = best;
      redi[2 * warp] = code;
      redi[2 * warp + 1] = anyneg_w != 0u;
    }
    sync();
    best = redd[0];
    code = redi[0];
    int neg = redi[1];
    for(int w = 1; w < NW; ++w)
    {
      const double ov = redd[w];
      const int oc = redi[2 * w];
      neg |= redi[2 * w + 1];
      if(ov < best || (ov == best && oc < code))
      {
        best = ov;
        code = oc;
      }
    }
    sync(); // the reduction scratch may be rewritten by the next call
    if(neg) return select_sequential(n, mc, nb, Cb, ldC, xs, bl, bu, xl, xu, stat);
    if(code == JRLQP_NONE) return {-1, ST_INACTIVE};
    return {code >> 3, code & 7};
  }

  // ------------------------------------------------------------------------------------------
  // computeStep_ (src/GoldfarbIdnaniSolver.cpp:136-148): d = J^T n+, z = J2 d2 (r and the Givens
  // recurrence follow on warps 0 and 1)
  // ------------------------------------------------------------------------------------------
  __device__ void compute_step(Sel sc)
  {
    const bool general = sc.st < ST_LOWER_BOUND;
    if(general)
      for(int i = tid; i < n; i += T) cv[i] = Cb[(long long)sc.p * ldC + i];
    if(rcols > 0) asm volatile("fence.proxy.async.global;" ::: "memory"); // (the last writes of J, before the barrier below)
    sync();
    if(rcols > 0 && tid == 0)
    {
      // the first chunks of z = J2 d2 travel while d is formed
      const int nch = (n - q + rcols - 1) / rcols;
      for(int k = 0; k < kRingStages - 1 && k < nch; ++k) ring_issue_up(q, k);
    }
    if(general)
    {
      // d, thread = column j of the column-major J: 32-byte vector loads down the column, DU of them (iterations) in flight;
      // 2 -> 4: config C cold +3.9 % (profiles/r5v_ab.txt), no spill. An L2 prefetch down the column lost 1 % (distance 128) and
      // 3 % (256) on config C (profiles/r5k_*).
      constexpr int DU = 4;
      for(int j = tid; j < n; j += T)
      {
        const double * Jj = Jc + (long long)j * ldl;
        double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        int i = 0;
#pragma unroll DU
        for(; i + 3 < n; i += 4)
        {
          const double2 p0 = *reinterpret_cast<const double2 *>(Jj + i);
          const double2 p1 = *reinterpret_cast<const double2 *>(Jj + i + 2);
          a0 = fma(p0.x, cv[i], a0);
          a1 = fma(p0.y, cv[i + 1], a1);
          a2 = fma(p1.x, cv[i + 2], a2);
          a3 = fma(p1.y, cv[i + 3], a3);
        }
        if(i < n) a0 = fma(Jj[i], cv[i], a0);
        if(i + 1 < n) a1 = fma(Jj[i + 1], cv[i + 1], a1);
        if(i + 2 < n) a2 = fma(Jj[i + 2], cv[i + 2], a2);
        double dj = (a0 + a1) + (a2 + a3);
        if(sc.st == ST_UPPER) dj = -dj;
        ds[j] = dj;
      }
    }
    else
    {
      const int pb = sc.p - mc; // +/- row pb of J
      for(int j = tid; j < n; j += T)
      {
        const double v = Jc[pb + (long long)j * ldl];
        ds[j] = sc.st == ST_UPPER_BOUND ? -v : v;
      }
    }
    sync();
    // z, thread = row i: z[i] = dot4_{j=q..n-1}(J(i,j), d[j]), accumulator (j-q)&3 — coalesced
    if(rcols > 0)
      z_ring();
    else
    for(int i = tid; i < n; i += T)
    {
      const double * Ji = Jc + i;
      double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
      int c = q;
#pragma unroll 2
      for(; c + 3 < n; c += 4)
      {
        const double j0 = Ji[(long long)c * ldl], j1 = Ji[(long long)(c + 1) * ldl], j2 = Ji[(long long)(c + 2) * ldl], j3 = Ji[(long long)(c + 3) * ldl];
        a0 = fma(j0, ds[c], a0);
        a1 = fma(j1, ds[c + 1], a1);
        a2 = fma(j2, ds[c + 2], a2);
        a3 = fma(j3, ds[c + 3], a3);
      }
      if(c < n) a0 = fma(Ji[(long long)c * ldl], ds[c], a0);
      if(c + 1 < n) a1 = fma(Ji[(long long)(c + 1) * ldl], ds[c + 1], a1);
      if(c + 2 < n) a2 = fma(Ji[(long long)(c + 2) * ldl], ds[c + 2], a2);
      zs[i] = (a0 + a1) + (a2 + a3);
    }
    sync();
  }

  // r = R^-1 d(0:q): column-oriented back substitution with true division, one warp
  __device__ void back_substitution()
  {
    for(int k = lane; k < q; k += 32) wv[k] = ds[k];
    __syncwarp();
#pragma unroll 1
    for(int k = q - 1; k >= 0; --k)
    {
      const double * Rk = Rp + colR(k);
      const double rk = wv[k] / Rk[k];
      __syncwarp();
      if(lane == 0) rs[k] = rk;
      for(int r = lane; r < k; r += 32) wv[r] = fma(-rk, Rk[r], wv[r]);
      __syncwarp();
    }
  }

  // computeStepLength_ (src/GoldfarbIdnaniSolver.cpp:150-219), incl. the activationStatus(k) quirk; one warp
  __device__ void step_length(Sel sc, double & t1, double & t2, int & l, double & nz, bool & zpos)
  {
    const double big = P.big_bnd;
    t1 = big;
    l = 0;
    {
      double bt = big;
      int bl_ = JRLQP_NONE;
      for(int k = lane; k < q; k += 32)
      {
        const int sk = stat[k]; // indexed by the position k, as in the reference (quirk, SURVEY §0)
        const double rk = rs[k];
        if(sk != ST_EQUALITY && sk != ST_FIXED && rk > 0.0)
        {
          const double tk = us[k] / rk;
          if(tk < bt)
          {
            bt = tk;
            bl_ = k;
          }
        }
      }
#pragma unroll
      for(int off = 16; off >= 1; off >>= 1)
      {
        const double ot = __shfl_xor_sync(JRLQP_FULL, bt, off);
        const int ol = __shfl_xor_sync(JRLQP_FULL, bl_, off);
        if(ot < bt || (ot == bt && ol < bl_))
        {
          bt = ot;
          bl_ = ol;
        }
      }
      bl_ = __shfl_sync(JRLQP_FULL, bl_, 0);
      bt = __shfl_sync(JRLQP_FULL, bt, 0);
      if(bl_ != JRLQP_NONE)
      {
        t1 = bt;
        l = bl_;
      }
    }
    double zz = 0.0;
    for(int k = lane; k < n; k += 32)
    {
      const double zk = zs[k];
      zz = fma(zk, zk, zz);
    }
    zpos = sqrt(warp_sum32(zz)) > 1e-14;

    t2 = big;
    double cz;
    if(sc.st < ST_LOWER_BOUND)
    {
      // lane t runs chain t of dot4(c, z), lane 4 + t chain t of dot4(c, x) (see gi_dense_cta.cuh)
      const double * v = (lane & 4) ? xs : zs;
      double acc = 0.0;
      if(lane < 8)
      {
#pragma unroll 2
        for(int k = lane & 3; k < n; k += 4) acc = fma(cv[k], v[k], acc);
      }
      const double a1 = __shfl_down_sync(JRLQP_FULL, acc, 1);
      const double s01 = acc + a1;
      const double s23 = __shfl_down_sync(JRLQP_FULL, s01, 2);
      const double dot = s01 + s23;
      cz = __shfl_sync(JRLQP_FULL, dot, 0);
      const double cx = __shfl_sync(JRLQP_FULL, dot, 4);
      nz = sc.st == ST_UPPER ? -cz : cz;
      if(zpos)
      {
        const double bb = sc.st == ST_UPPER ? bu[sc.p] : bl[sc.p]; // EQUALITY: bl (addInitialConstraint)
        t2 = (bb - cx) / cz;
      }
    }
    else
    {
      const int pb = sc.p - mc;
      cz = zs[pb];
      nz = sc.st == ST_UPPER_BOUND ? -cz : cz;
      if(zpos)
      {
        const double bb = sc.st == ST_UPPER_BOUND ? xu[pb] : xl[pb];
        t2 = (bb - xs[pb]) / cz;
      }
    }
  }

  // x += t z ; f += t (n+.z) (t/2 + u[q]) ; u(0:q) -= t r ; u[q] += t — one warp
  __device__ void take_step(double t, double nz, bool primal)
  {
    const double uq = us[q];
    __syncwarp();
    if(primal)
    {
      for(int r = lane; r < n; r += 32) xs[r] = fma(t, zs[r], xs[r]);
      f += (t * nz) * (0.5 * t + uq);
    }
    for(int k = lane; k < q; k += 32) us[k] = fma(-t, rs[k], us[k]);
    if(lane == 0) us[q] = uq + t;
    __syncwarp();
  }

  // addConstraint (src/DualSolver.cpp:231-235) + addConstraint_ (src/GoldfarbIdnaniSolver.cpp:221-237):
  // apply the rotation table, thread = row of J (coalesced in the column-major storage)
  __device__ void add_constraint()
  {
    q += 1;
    const int lo = q - 1;
    if(lo <= n - 2 && rcols > 0)
      add_rotations_ring(lo);
    else if(lo <= n - 2)
    {
      for(int row = tid; row < n; row += T)
      {
        double * Ji = Jc + row;
        double y = Ji[(long long)(n - 1) * ldl];
        int i = n - 2;
        double xv[PF];
        if(i - (PF - 1) >= lo)
        {
#pragma unroll
          for(int u = 0; u < PF; ++u) xv[u] = Ji[(long long)(i - u) * ldl];
        }
#pragma unroll 1
        while(i - (PF - 1) >= lo)
        {
          double xn[PF];
          const bool more = i - (2 * PF - 1) >= lo;
          if(more)
          {
#pragma unroll
            for(int u = 0; u < PF; ++u) xn[u] = Ji[(long long)(i - PF - u) * ldl];
          }
          double o[PF];
#pragma unroll
          for(int u = 0; u < PF; ++u)
          {
            const double2 cs2 = gcs[i - u];
            const double c = cs2.x, sn = cs2.y, xi = xv[u];
            o[u] = fma(c, y, sn * xi);
            y = fma(c, xi, -(sn * y));
          }
#pragma unroll
          for(int u = 0; u < PF; ++u) Ji[(long long)(i - u + 1) * ldl] = o[u];
          i -= PF;
          if(more)
          {
#pragma unroll
            for(int u = 0; u < PF; ++u) xv[u] = xn[u];
          }
        }
#pragma unroll 1
        for(; i >= lo; --i)
        {
          const double2 cs2 = gcs[i];
          const double c = cs2.x, sn = cs2.y;
          const double xi = Ji[(long long)i * ldl];
          Ji[(long long)(i + 1) * ldl] = fma(c, y, sn * xi);
          y = fma(c, xi, -(sn * y));
        }
        Ji[(long long)lo * ldl] = y;
      }
    }
    // R(0:q, q-1) = d(0:q), with d[q-1] = rho
    for(int k = tid; k < q; k += T) Rp[colR(q - 1) + k] = k == q - 1 ? scr[10] : ds[k];
    sync();
  }

  // removeConstraint (src/DualSolver.cpp:237-244) + removeConstraint_ (src/GoldfarbIdnaniSolver.cpp:239-256), whole CTA
  __device__ void remove_constraint(int l)
  {
    sync();
    // u.segment(l, q-l) = u.tail(q-l) (u has q+1 entries) ; A_.deactivate(l)
    const int removed = alist[l];
    {
      // shift through the work vector wv / the Givens kind array gk (free here)
      for(int k = l + tid; k < q; k += T) wv[k] = us[k + 1];
      for(int k = l + tid; k + 1 < q; k += T) gk[k] = alist[k + 1];
      sync();
      for(int k = l + tid; k < q; k += T) us[k] = wv[k];
      for(int k = l + tid; k + 1 < q; k += T) alist[k] = gk[k];
      if(tid == 0) stat[removed] = ST_INACTIVE;
    }
    const int qn = q - 1;
    sync();
#pragma unroll 1
    for(int i = l; i < qn; ++i)
    {
      double * Ri = Rp + colR(i);
      double * Ri1 = Rp + colR(i + 1);
      for(int k = tid; k < i; k += T) Ri[k] = Ri1[k];
      double c, sn, r;
      make_givens(Ri1[i], Ri1[i + 1], c, sn, r);
      if(tid == 0) Ri[i] = r;
      // rows i, i+1 of columns i+2 .. q (thread = column)
      for(int j = i + 2 + tid; j <= qn; j += T)
      {
        double * Rj = Rp + colR(j);
        const double xi = Rj[i], yi = Rj[i + 1];
        Rj[i] = fma(c, xi, -(sn * yi));
        Rj[i + 1] = fma(c, yi, sn * xi);
      }
      // columns i, i+1 of J (thread = row)
      for(int row = tid; row < n; row += T)
      {
        double * Ji = Jc + row + (long long)i * ldl;
        const double xi = Ji[0], yi = Ji[ldl];
        Ji[0] = fma(c, xi, -(sn * yi));
        Ji[ldl] = fma(c, yi, sn * xi);
      }
      sync();
    }
    q -= 1;
    sync();
  }

#include "gi_large_warm.inl"

  // ------------------------------------------------------------------------------------------
  // DualSolver::solve (src/DualSolver.cpp:91-168) for problem b, initActiveSet / addInitialConstraint
  // (src/GoldfarbIdnaniSolver.cpp:268-338) folded into the same loop (see gi_dense_cta.cuh)
  // ------------------------------------------------------------------------------------------
  __device__ void solve(long long b)
  {
    bl = P.bl + b * P.sbl;
    bu = P.bu + b * P.sbu;
    xl = nb ? P.xl + b * P.sxl : nullptr;
    xu = nb ? P.xu + b * P.sxu : nullptr;
    Cb = P.C + b * P.sC;
    ldC = P.ldc;
    cvec = ((reinterpret_cast<unsigned long long>(Cb) & 15ull) == 0ull) && ((ldC & 1) == 0);

    int it = 0;
    int cursor = 0;
    if(WARM)
    {
      const int st0 = init_warm(b, it);
      if(st0 != TS_SUCCESS)
      {
        write_failure(b, st0);
        return;
      }
      cursor = m;
    }
    else if(!init(b))
    {
      write_failure(b, TS_NON_POS_HESSIAN);
      return;
    }

    int status = TS_MAX_ITER_REACHED;
    bool skip = false;
    Sel sc{-1, ST_INACTIVE};
    const double big = P.big_bnd;
    int * dec = iscr; // [0] add, [1] l, [2] status on break (-1: none)
    double * decd = scr + 13; // [0] f
#pragma unroll 1
    for(;;)
    {
      bool pre = false;
      while(cursor < m)
      {
        const int c = cursor++;
        if(eqf[c])
        {
          sc = {c, c < mc ? ST_EQUALITY : ST_FIXED};
          pre = true;
          break;
        }
      }
      if(pre && q >= n)
      {
        // more than nbVar equalities / fixed variables (the reference would write past its workspaces)
        write_failure(b, TS_OVERCONSTRAINED_PROBLEM);
        return;
      }
      if(!pre)
      {
        if(it >= P.max_iter) break; // MAX_ITER_REACHED
        if(!skip)
        {
          sc = select();
          if(sc.st == ST_INACTIVE)
          {
            status = TS_SUCCESS;
            break;
          }
        }
      }
      if(pre || !skip)
      {
        if(tid == 0) us[q] = 0.0; // published by the barriers of compute_step
      }
      compute_step(sc);
      if(warp == 0)
      {
        back_substitution();
        double t1, t2, nz;
        int l;
        bool zpos;
        step_length(sc, t1, t2, l, nz, zpos);
        double t;
        bool primal = true, add = true;
        int brk = -1;
        if(pre)
          t = zpos ? t2 : 0.0; // exact step onto the constraint (src/GoldfarbIdnaniSolver.cpp:307-322)
        else
        {
          t = t2 < t1 ? t2 : t1; // std::min(t1, t2)
          if(t >= big)
            brk = TS_INFEASIBLE;
          else if(t2 >= big)
            primal = add = false; // dual-only step, then drop
          else
            add = t == t2; // full step -> add ; partial step -> drop
        }
        if(brk < 0)
        {
          take_step(t, nz, primal);
          if(add && lane == 0)
          {
            alist[q] = sc.p; // DualSolver::addConstraint bookkeeping (src/DualSolver.cpp:231-235)
            stat[sc.p] = (signed char)sc.st;
          }
        }
        if(lane == 0)
        {
          dec[0] = add;
          dec[1] = l;
          dec[2] = brk;
          decd[0] = f;
        }
      }
      else if(warp == 1)
        givens_chain(q, n, lane, ds, gcs, gc, gs, gk, scr, reinterpret_cast<double *>(gcs) + ((n + 3) & ~3));
      sync();
      const bool add = dec[0] != 0;
      const int l = dec[1];
      const int brk = dec[2];
      f = decd[0];
      if(brk >= 0)
      {
        status = brk;
        break;
      }
      if(add)
        add_constraint();
      else
        remove_constraint(l);
      if(!pre)
      {
        skip = !add;
        ++it;
      }
    }
    sync();
    write_result(b, status, it);
  }

  __device__ void write_result(long long b, int status, int it)
  {
    double * xo = P.x + b * n;
    for(int i = tid; i < n; i += T) xo[i] = xs[i];
    if(P.u)
    {
      // DualSolver::multipliers (src/DualSolver.cpp:38-69): zero, then scatter the condensed multipliers
      double * uo = P.u + b * m;
      for(int i = tid; i < m; i += T) uo[i] = 0.0;
      sync();
      for(int k = tid; k < q; k += T)
      {
        const int i = alist[k];
        const int s = stat[i];
        uo[i] = (s == ST_UPPER || s == ST_UPPER_BOUND) ? us[k] : -us[k];
      }
    }
    if(P.active_set)
    {
      signed char * ao = P.active_set + b * m;
      for(int i = tid; i < m; i += T) ao[i] = stat[i];
    }
    if(P.active_list)
    {
      int * lo = P.active_list + b * n;
      for(int k = tid; k < n; k += T) lo[k] = k < q ? alist[k] : -1;
    }
    if(tid == 0)
    {
      if(P.f) P.f[b] = f;
      if(P.iterations) P.iterations[b] = it;
      if(P.status) P.status[b] = status;
      if(P.n_active) P.n_active[b] = q;
    }
  }

  __device__ void write_failure(long long b, int status)
  {
    double * xo = P.x + b * n;
    for(int i = tid; i < n; i += T) xo[i] = 0.0;
    if(P.u)
      for(int i = tid; i < m; i += T) P.u[b * m + i] = 0.0;
    if(P.active_set)
      for(int i = tid; i < m; i += T) P.active_set[b * m + i] = ST_INACTIVE;
    if(P.active_list)
      for(int k = tid; k < n; k += T) P.active_list[b * n + k] = -1;
    if(tid == 0)
    {
      if(P.f) P.f[b] = 0.0;
      if(P.iterations) P.iterations[b] = 0;
      if(P.status) P.status[b] = status;
      if(P.n_active) P.n_active[b] = 0;
    }
  }
};

// Persistent kernel: every CTA claims one workspace slice (atomic flag per slice: launches of the same
// solver may overlap on different streams; resident CTAs never outnumber the slices) and pulls
// problem indices from the ticket counter.
template<int T, bool WARM>
__global__ void __launch_bounds__(T, 2) gi_large_kernel(const GiParams p)
{
  extern __shared__ __align__(16) double smem[];
  __shared__ unsigned long long ticket;
  __shared__ int slot_s;
  if(threadIdx.x == 0)
  {
    int i = (int)(blockIdx.x % (unsigned)p.work_slots);
    while(atomicCAS(p.work_busy + i, 0, 1) != 0) i = i + 1 == p.work_slots ? 0 : i + 1;
    __threadfence();
    slot_s = i;
  }
  __syncthreads();
  const int slot = slot_s;
  GiLarge<T, WARM> cta(p, smem, p.work + (long long)slot * p.work_stride);
  cta.ring_setup();
  for(;;)
  {
    __syncthreads();
    if(threadIdx.x == 0) ticket = atomicAdd(p.counter, 1ull);
    __syncthreads();
    const unsigned long long b = ticket;
    if(b >= (unsigned long long)p.batch) break;
    cta.solve((long long)b);
  }
  __syncthreads();
  if(threadIdx.x == 0)
  {
    __threadfence();
    atomicExch(p.work_busy + slot, 0);
  }
}

// Transposed copy of a batch-shared C (n x mc column-major, one normal per column) for the coalesced constraint scan of
// the large-n kernel (layout: groups of 128 constraints, see ct_offset), 32 x 32 tiles through shared memory.
__global__ void __launch_bounds__(256) transpose_c_kernel(const double * __restrict__ C, int ldc, int n, int mc, double * __restrict__ Ct)
{
  __shared__ double tile[32][33];
  const int c0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; // 32 x 8
  for(int r = ty; r < 32; r += 8)
  {
    const int c = c0 + r, k = k0 + tx;
    tile[r][tx] = (c < mc && k < n) ? C[(long long)c * ldc + k] : 0.0;
  }
  __syncthreads();
  for(int r = ty; r < 32; r += 8)
  {
    const int k = k0 + r, c = c0 + tx;
    if(k < n && c < mc) Ct[ct_offset(c, n) + (long long)k * JRLQP_CT_LD] = tile[tx][r];
  }
}

// Factor of a batch-shared G for the large-n kernel: ONE CTA runs the same Cholesky / J = L^-T code as the solver
// CTAs (same bits) and leaves L, J (column-major), diag(L) and its reciprocals in `pre` (layout: gi_params.h).
template<int T>
__global__ void __launch_bounds__(T, 1) gi_large_prefactor_kernel(const GiParams p, double * pre, int * pre_ok)
{
  extern __shared__ __align__(16) double smem[];
  GiLarge<T, false> cta(p, smem, pre); // p.L == nullptr, p.pre == nullptr (set by the host)
  const int n = p.n, ldl = (n + 3) & ~3, nv = (n + 3) & ~3;
  const bool ok = cta.cholesky(0);
  if(!ok)
  {
    if(threadIdx.x == 0) *pre_ok = 0;
    return;
  }
  double * Lk = pre + 2ll * n * ldl;
  double * pd = pre + 3ll * n * ldl;
  for(long long e = threadIdx.x; e < (long long)n * ldl; e += T) Lk[e] = cta.Lw[e];
  for(int i = threadIdx.x; i < n; i += T)
  {
    pd[i] = cta.ldiag[i];
    pd[nv + i] = cta.rinv[i];
  }
  __syncthreads();
  cta.build_J(0);
  __syncthreads();
  cta.transpose_J();
  if(threadIdx.x == 0) *pre_ok = 1;
}

} // namespace jrlqp
