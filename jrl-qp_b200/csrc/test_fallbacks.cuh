// Test-only instrumentation of the stock-arithmetic fallbacks (build with -DJRLQP_TEST_FALLBACKS; never in the shipped
// library, where every macro below expands to nothing and the kernels are unchanged instruction for instruction).
//
// The serial recurrences prove each fast quotient / square root correctly rounded and, when a proof is declined, redo
// the work with the stock `/` and `sqrt` (fp64_exact.cuh). Ordinary inputs rarely decline a proof, so the recovery
// code would otherwise be checked by reading only. In the test build:
//  * fb_hits[site] counts the fallbacks taken at each site (one increment per fallback, from one lane);
//  * fb_decline_all != 0 makes every proof decline (div_rcp, div_proof, the inline proofs of the Givens recurrences,
//    the vote of the small-tile LLT, the branch-free check of the four-warp recurrence), so that every fallback runs
//    on every input and its results can be compared with the oracle bit for bit.
// Each translation unit has its own copy of both (no relocatable device code): the host functions of capi.cu,
// structured.cu and blockgi.cu read and set their unit's copy; capi.cu exports one call for all three
// (jrlqp_test_fallback_counts / jrlqp_test_fallback_decline_all).
#pragma once

namespace jrlqp
{

enum FallbackSite
{
  FB_GI_X = 0,          // x = -G^-1 a of the dense kernel: stock division after a declined div_rcp
  FB_GIVENS_LINK = 1,   // givens_link_slow: stock division when the quotient from the precomputed 1 / p is not proven
  FB_CHAIN_CAREFUL = 2, // givens_chain: the chain redone literally after a declined deferred proof
  FB_BACKSUB = 3,       // back_substitution_exact after a declined proof
  FB_REC_CAREFUL = 4,   // GiCta::givens_recurrence: the careful pass after a declined deferred proof
  FB_REC_BAD = 5,       // GiCta::givens_recurrence, W = 4: a link predicted on the fast branch was not
  FB_LARGE_INIT = 6,    // initial_point_blocked of the large kernel: stock division
  FB_WARM_B = 7,        // warm start, B = L^-1 N: stock division
  FB_BLOCK_SOLVE = 8,   // TriWarpSolver: block_solve_exact after block_solve_fast failed (structured solves and BlockGI)
  FB_R_SOLVE = 9,       // BlockGI r_solve_blocked: one link at a time after an unproven quotient
  FB_LLT_SMALL = 10,    // small-tile LLT: stock sqrt and divisions after a failed per-column vote
  FB_NSITES = 11
};

#ifdef JRLQP_TEST_FALLBACKS
__device__ unsigned long long fb_hits[FB_NSITES];
__device__ int fb_decline_all;

// host side, per translation unit: add the unit's counts to out[FB_NSITES] and clear them; set the decline flag
static inline int fb_collect(unsigned long long * out)
{
  unsigned long long h[FB_NSITES];
  cudaError_t e = cudaMemcpyFromSymbol(h, fb_hits, sizeof(h));
  if(e != cudaSuccess) return (int)e;
  for(int s = 0; s < FB_NSITES; ++s) out[s] += h[s];
  for(int s = 0; s < FB_NSITES; ++s) h[s] = 0;
  return (int)cudaMemcpyToSymbol(fb_hits, h, sizeof(h));
}
static inline int fb_set_decline(int on)
{
  return (int)cudaMemcpyToSymbol(fb_decline_all, &on, sizeof(on));
}
#  define JRLQP_FB_HIT(site) atomicAdd(&::jrlqp::fb_hits[::jrlqp::site], 1ull)
#  define JRLQP_FB_HIT_IF(cond, site) \
    do                                \
    {                                 \
      if(cond) JRLQP_FB_HIT(site);    \
    } while(0)
#  define JRLQP_FB_DECLINE(ok) ok = (ok) && ::jrlqp::fb_decline_all == 0 // a proof fails under the decline flag
#  define JRLQP_FB_FORCE(bad) bad = (bad) || ::jrlqp::fb_decline_all != 0 // a check fails under the decline flag
#else
#  define JRLQP_FB_HIT(site) ((void)0)
#  define JRLQP_FB_HIT_IF(cond, site) ((void)0)
#  define JRLQP_FB_DECLINE(ok) ((void)0)
#  define JRLQP_FB_FORCE(bad) ((void)0)
#endif

} // namespace jrlqp
