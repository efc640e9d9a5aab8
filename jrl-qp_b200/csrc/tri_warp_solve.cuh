// Warp-level triangular solves with the structured Cholesky factor of a tri-block-diagonal chain of uniform dense tiles
// (NB = 8 / 12 / 16 rows, dense tiles at 16-byte aligned offsets: the MPC shape of BASELINE.json config 5). Used by the
// structured solver (blockgi.cuh: the two solves of every iteration) and by the batch solve entry points
// (structured.cu: jrlqp_structured_solve_*), in place of the CTA-wide sg_solve_inplace of structured.cuh.
//
// Replaces decomposition::triBlockDiagLSolve / triBlockDiagLTransposeSolve (src/decomposition/triBlockDiagLLT.cpp:38-158)
// behind structured::StructuredG::solveL / solveInPlaceLTranspose (src/structured/StructuredG.cpp:45-113), hints included.
#pragma once

#include "fp64_exact.cuh"

#include <cuda_runtime.h>
#include <stdint.h>

namespace jrlqp
{

#define TW_FULL 0xffffffffu

// 1 / d to a few ulps from the hardware seed (3 Newton steps): the reciprocal a proven quotient starts from
// (fp64_exact.cuh div_rcp: the result never depends on it)
__device__ __forceinline__ double bg_rcp(double d)
{
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  double e = fma(-d, r, 1.0);
  r = fma(r, e, r);
  e = fma(-d, r, 1.0);
  r = fma(r, e, r);
  e = fma(-d, r, 1.0);
  return fma(r, e, r);
}

__device__ __forceinline__ unsigned bg_smem_addr(const void * p)
{
  return (unsigned)__cvta_generic_to_shared(p);
}


// State of one warp: a RING-deep stage of tile pairs (diagonal tile, sub-diagonal tile) in shared memory filled by TMA bulk
// copies, one mbarrier per stage, the (L_kk, ~ 1 / L_kk) pairs of the staged diagonal tiles, the block offsets.
struct TriWarp
{
  static constexpr int RING = 3, AHEAD = RING - 1;
  double * ring; // [RING][2][NB * LDT], 16-byte aligned
  double2 * dgp; // [RING][16]
  unsigned long long * bars; // [RING], initialised by init_barriers()
  const long long *sdoff, *sooff; // offsets of the diagonal / sub-diagonal blocks inside an instance
  const double * base; // the instance
  int b, n, lane;
  unsigned rph; // phase parities of the barriers (bit = stage), tracked by every lane

  static __host__ __device__ int ring_ld(int nb) { return nb == 16 ? 18 : nb; } // (16: padded columns, 16-way bank conflicts otherwise)
  // doubles of shared memory per warp: tiles + pairs (the barriers take RING more 8-byte words)
  static __host__ __device__ long long ring_doubles(int nb) { return nb ? (long long)RING * 2 * nb * ring_ld(nb) + RING * 32 : 0; }

  __device__ void init_barriers() const // one thread; followed by a barrier of the threads that use them
  {
    for(int i = 0; i < RING; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bg_smem_addr(bars + i)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }

  // ------------------------------------------------------------------------------------------------------------
  // Structured solves on ONE WARP for tri-block-diagonal chains of uniform dense tiles (P.fast_nb = 8 / 12 / 16; the MPC
  // shape of BASELINE.json config 5). Round 1 ran sg_solve_inplace on the whole CTA: a tile load from L2 / HBM and two
  // block barriers per column, with one true division every thread repeats — half of a solve (profiles/r02y_*). Here
  //   * lane r owns row r of the block; the substitution is the uniform-pivot recurrence of the dense kernel: every lane
  //     applies link k's update to the NEXT pivot itself (same fma, same operands as the lane that owns it), so a link is
  //     one quotient + one fma on the dependent chain and every x_k ends up uniform in registers — the product with the
  //     sub-diagonal tile of the next block needs no exchange at all;
  //   * the quotient w_k / L_kk comes from a reciprocal prepared one block ahead and is PROVEN correctly rounded
  //     (fp64_exact.cuh); a block with an unproven quotient is redone with true divisions;
  //   * the tiles of the next RING - 1 blocks are in flight as TMA bulk copies (cp.async.bulk, completion on an mbarrier per
  //     stage) while a block is solved; the other warps of the CTA wait at the closing barrier.
  // Per-output operation order = structured.cuh / oracle/decomp_oracle.cpp (dot4 for the tile products, column-oriented
  // substitution), hence the same bits. v: the vector in shared memory; hints as sg_solve_inplace.
  // ------------------------------------------------------------------------------------------------------------
  template<int NB>
  __device__ __forceinline__ void ring_issue(const int i, const int is, const int slot)
  {
    // tiles of diagonal block i and (is >= 0) sub-diagonal block is into stage `slot`; lane 0 only
    constexpr int LDT = NB == 16 ? 18 : NB, TT = NB * LDT;
    double * Ls = ring + slot * 2 * TT;
    const unsigned bar = bg_smem_addr(bars + slot);
    const unsigned bytes = (is >= 0 ? 2u : 1u) * NB * NB * 8u;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // earlier generic reads of this stage are done
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    for(int t = 0; t < (is >= 0 ? 2 : 1); ++t)
    {
      const double * src = base + (t == 0 ? sdoff[i] : sooff[is]);
      double * dst = Ls + t * TT;
      if(LDT == NB)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(bg_smem_addr(dst)), "l"(src),
                     "r"(NB * NB * 8u), "r"(bar)
                     : "memory");
      else
        for(int c = 0; c < NB; ++c)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(bg_smem_addr(dst + c * LDT)),
                       "l"(src + c * NB), "r"(NB * 8u), "r"(bar)
                       : "memory");
    }
  }

  __device__ __forceinline__ void ring_wait(const int slot)
  {
    unsigned done = 0;
    const unsigned bar = bg_smem_addr(bars + slot), par = (rph >> slot) & 1u;
    while(!done)
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(done) : "r"(bar), "r"(par) : "memory");
    rph ^= 1u << slot;
  }

  // links [klo, khi) of the substitution with true divisions, one shuffle per link (partial first blocks, and the rare
  // block whose fast quotients could not be proven)
  template<int NB, bool TR>
  __device__ __noinline__ double block_solve_exact(const double * Ls, double wr, const int klo, const int khi)
  {
    constexpr int LDT = NB == 16 ? 18 : NB;
    const int lc = min(lane, NB - 1);
#pragma unroll 1
    for(int s = 0; s < khi - klo; ++s)
    {
      const int k = TR ? khi - 1 - s : klo + s;
      const double xk = __shfl_sync(TW_FULL, wr, k) / Ls[k + k * LDT];
      const double lr = TR ? Ls[k + lc * LDT] : Ls[lc + k * LDT];
      const double nw = fma(-xk, lr, wr);
      const bool upd = TR ? lane < k : (lane > k && lane < NB);
      wr = lane == k ? xk : (upd ? nw : wr);
    }
    return wr;
  }

  // the whole block, uniform-pivot recurrence: per link one pair load (L_kk and its reciprocal, prepared a block ahead),
  // three FMAs for the quotient, one for the next pivot, one (predicated) for the lane's own row — straight-line code.
  // A lane stops updating its row at its own link, so lane k is left holding ITS PIVOT: after the loop it forms its own
  // quotient again (the same three FMAs on the same operands as the uniform copy: the same bits), PROVES it correctly
  // rounded (fp64_exact.cuh) and keeps it as its entry of the solution. false: some proof failed, wr and xs are to be
  // discarded.
  template<int NB, bool TR>
  __device__ __forceinline__ bool block_solve_fast(const double * Ls, const double2 * dp, double & wr, double (&xs)[NB])
  {
    constexpr int LDT = NB == 16 ? 18 : NB;
    const int lc = min(lane, NB - 1);
    double wp = __shfl_sync(TW_FULL, wr, TR ? NB - 1 : 0);
#pragma unroll
    for(int s = 0; s < NB; ++s)
    {
      const int k = TR ? NB - 1 - s : s;
      const int kn = TR ? k - 1 : k + 1; // the next pivot
      const double tn = s + 1 < NB ? __shfl_sync(TW_FULL, wr, kn) : 0.0; // w_kn before this link's update
      const double2 dr = dp[k];
      const double q0 = wp * dr.y;
      const double e = fma(-dr.x, q0, wp);
      const double xk = fma(e, dr.y, q0);
      xs[k] = xk;
      if(s + 1 < NB) wp = fma(-xk, TR ? Ls[k + kn * LDT] : Ls[kn + k * LDT], tn);
      const double lr = TR ? Ls[k + lc * LDT] : Ls[lc + k * LDT];
      if(TR ? lane < k : lane > k) wr = fma(-xk, lr, wr);
    }
    const double2 own = dp[lc];
    const double q0 = wr * own.y;
    const double e = fma(-own.x, q0, wr);
    const double xo = fma(e, own.y, q0);
    const bool ok = lane >= NB || div_proof(wr, own.x, xo);
    wr = xo;
    return __all_sync(TW_FULL, ok);
  }

  template<int NB, bool TR>
  __device__ void solve(double * v, const int start, int end)
  {
    constexpr int LDT = NB == 16 ? 18 : NB, TT = NB * LDT;
    static_assert(NB % 4 == 0 && NB <= 16, "tile size");
    const int lc = min(lane, NB - 1);
    if(end < 0) end = n;
    // blocks in processing order: forward i0, i0 + 1, ... (the first block the hint start touches, then all that follow);
    // transposed i1, i1 - 1, ..., 0 (the first block below the hint end)
    int first, cnt;
    if(!TR)
    {
      first = max(0, (start + NB - 1) / NB - 1);
      cnt = b - first;
    }
    else
    {
      if(end <= 0) return;
      first = min(b - 1, (end - 1) / NB);
      cnt = first + 1;
    }
    auto blk = [&](int j) { return TR ? first - j : first + j; };
    auto issue = [&](int j)
    {
      if(lane == 0)
      {
        const int i = blk(j);
        ring_issue<NB>(i, j == 0 ? -1 : (TR ? i : i - 1), j % RING);
      }
    };
    // (L_kk, ~ 1 / L_kk) of the tile in stage `slot`, lane k the pair k
    auto prepare = [&](int slot)
    {
      const double dgv = (ring + slot * 2 * TT)[lc + lc * LDT];
      if(lane < NB) dgp[slot * 16 + lane] = make_double2(dgv, bg_rcp(dgv));
    };
    __syncwarp();
    for(int j = 0; j < AHEAD && j < cnt; ++j) issue(j);
    ring_wait(0);
    prepare(0);
    double xs[NB];
#pragma unroll
    for(int k = 0; k < NB; ++k) xs[k] = 0.0;
    double wnx = v[blk(0) * NB + lc]; // the block's entries of the vector, fetched one block ahead (v may live in global memory)
#pragma unroll 1
    for(int j = 0; j < cnt; ++j)
    {
      const int i = blk(j);
      const int slot = j % RING;
      const double * Ls = ring + slot * 2 * TT;
      const double * Ss = Ls + TT;
      __syncwarp(); // every lane is done with the stage of block j - 1, which the next copy overwrites; pairs of block j visible
      if(j + AHEAD < cnt) issue(j + AHEAD);
      if(j + 1 < cnt)
      {
        ring_wait((j + 1) % RING);
        prepare((j + 1) % RING);
      }
      double wr = wnx;
      if(j + 1 < cnt) wnx = v[blk(j + 1) * NB + lc];
      if(j > 0)
      {
        // forward: w -= S_{i-1} x_{i-1} (S(r, k) at Ss[r + k LDT]); transposed: w -= S_i^T x_{i+1} (S(k, r) at Ss[k + r LDT])
        double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll
        for(int k = 0; k < NB; k += 4)
        {
          c0 = fma(TR ? Ss[k + lc * LDT] : Ss[lc + k * LDT], xs[k], c0);
          c1 = fma(TR ? Ss[k + 1 + lc * LDT] : Ss[lc + (k + 1) * LDT], xs[k + 1], c1);
          c2 = fma(TR ? Ss[k + 2 + lc * LDT] : Ss[lc + (k + 2) * LDT], xs[k + 2], c2);
          c3 = fma(TR ? Ss[k + 3 + lc * LDT] : Ss[lc + (k + 3) * LDT], xs[k + 3], c3);
        }
        wr = wr - ((c0 + c1) + (c2 + c3));
      }
      // hints: only the first block can be partial (forward: rows from `start` on; transposed: rows before `end`)
      int klo = 0, khi = NB;
      if(j == 0)
      {
        if(!TR)
          klo = max(0, start - i * NB);
        else
          khi = min(NB, end - i * NB);
      }
      const double w0 = wr;
      bool fast = klo == 0 && khi == NB;
      if(fast)
      {
        fast = block_solve_fast<NB, TR>(Ls, dgp + slot * 16, wr, xs);
        JRLQP_FB_HIT_IF(!fast && lane == 0, FB_BLOCK_SOLVE);
      }
      if(!fast)
      {
        wr = block_solve_exact<NB, TR>(Ls, w0, klo, khi);
#pragma unroll
        for(int k = 0; k < NB; ++k) xs[k] = __shfl_sync(TW_FULL, wr, k);
      }
      if(lane < NB) v[i * NB + lane] = wr;
    }
  }

};

} // namespace jrlqp
