// Host side of the structured solver's C-ABI (include/jrlqp_b200.h, jrlqp_blockgi_*): descriptor upload,
// workspace sizing, the factorisation + solver launches, and the host-pointer entry point. Pure CUDA runtime.
#include "smem_limit.hpp"
#include "blockgi.cuh"
#include "structured_host.hpp"

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <string>
#include <vector>

using namespace jrlqp;

namespace jrlqp
{
void count_launch(); // capi.cu: feeds jrlqp_launch_count()

} // namespace jrlqp

struct jrlqp_blockgi
{
  jrlqp_structured * g = nullptr; // owns the structure of G (descriptor on the device, launch configuration)
  int n = 0, mc = 0, nb = 0, cb = 0;
  long long capacity = 0;
  int device = 0;
  jrlqp_options opt{500, 1e100, 0, 0};
  std::vector<int> cnvar, cncstr, cld, cvar0, ccstr0, toblock;
  std::vector<long long> coff;
  long long c_min_stride = 0;
  int *d_cnvar = nullptr, *d_cld = nullptr, *d_cvar0 = nullptr, *d_ccstr0 = nullptr, *d_toblock = nullptr;
  long long * d_coff = nullptr;
  // launch configuration (depends on max_iter through the record table)
  int smem = 0, occ = 0, grid = 0, configured_iter = -1;
  // workspace
  double * d_ws = nullptr;
  long long ws_stride = 0, qcap = 0, ws_slots = 0;
  unsigned long long * d_ticket = nullptr;
  int * d_ok = nullptr;
  long long ok_cap = 0;
  double * d_gshared = nullptr; // private copy of a shared (stride 0) G, factorised once per call
  // host staging
  double * d_in = nullptr;
  long long d_in_bytes = 0;
  unsigned char * d_out = nullptr;
  long long d_out_bytes = 0;
  cudaStream_t stream = nullptr;
  int bthreads = 0; // threads per CTA of blockgi_kernel (the structured kernels keep s->g->threads)
  int flags = 7; // BGF_* fast paths (blockgi.cuh); JRLQP_BLOCKGI_FAST overrides
  int fast_nb = 0; // uniform dense tile size of a tri-block-diagonal G (8 / 12 / 16), else 0
  void (*kernel)(const BlockGiParams) = nullptr;
  std::string err;

  bool check(cudaError_t e, const char * what)
  {
    if(e == cudaSuccess) return true;
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
  }
};

namespace
{

int configure(jrlqp_blockgi * s)
{
  if(s->configured_iter == s->opt.max_iter) return JRLQP_OK;
  cudaDeviceProp prop;
  SCK(cudaGetDeviceProperties(&prop, s->device));
  const int m = s->mc + s->nb;
  s->fast_nb = s->g->small_nb;
  s->flags = 7;
  if(const char * e = getenv("JRLQP_BLOCKGI_FAST")) s->flags = atoi(e) & 7;
  s->kernel = s->n <= 512 ? blockgi_kernel<4> : blockgi_kernel<8>; // entries of a reflector per thread: 128 classes x 4 / 8
  const long long smem = BlockGi<8>::smem_bytes(s->n, s->g->nmax, m, std::max(1, s->opt.max_iter), s->fast_nb, s->g->b);
  if(smem > (long long)prop.sharedMemPerBlockOptin)
  {
    s->err = "problem does not fit in shared memory (n, block size or max_iter too large)";
    return JRLQP_ERR_ARG;
  }
  s->smem = (int)smem;
  if(s->bthreads == 0)
  {
    s->bthreads = 128; // one class of the reflector products per thread (blockgi.cuh); the kernel is compiled for 128 threads
  }
  SCK(jrlqp::raise_smem_limit(s->kernel, s->smem));
  SCK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s->occ, s->kernel, s->bthreads, s->smem));
  if(s->occ < 1)
  {
    s->err = "kernel cannot be made resident";
    return JRLQP_ERR_ARG;
  }
  s->grid = s->occ * s->g->num_sms;
  // record storage: one record per iteration at most, a Householder vector of <= n doubles or a Givens
  // sequence of <= 2 (n - 1); the active set holds at most n constraints, so the sum of the lengths of the
  // reflectors alive at any time is bounded, but dropped ones stay in the sequence (as in the reference)
  s->qcap = (long long)std::max(1, s->opt.max_iter) * 2 * s->n;
  const long long stride = (long long)s->n * (s->n + 1) / 2 + s->qcap;
  if(stride != s->ws_stride || s->ws_slots < s->grid)
  {
    if(s->d_ws) cudaFree(s->d_ws);
    s->d_ws = nullptr;
    s->ws_stride = stride;
    s->ws_slots = s->grid;
    SCK(cudaMalloc(&s->d_ws, sizeof(double) * stride * s->grid));
  }
  s->configured_iter = s->opt.max_iter;
  return JRLQP_OK;
}

} // namespace

extern "C"
{

int jrlqp_blockgi_create(jrlqp_blockgi ** out, const jrlqp_structure * G, const jrlqp_cstructure * C, int32_t use_bounds,
                         int64_t batch_capacity, int32_t device)
{
  if(!out) return JRLQP_ERR_ARG;
  *out = nullptr;
  if(!G || !C || C->nblocks < 0 || batch_capacity < 0) return JRLQP_ERR_ARG;
  if(C->nblocks > 0 && (!C->nvar || !C->ncstr || !C->offset || !C->ld)) return JRLQP_ERR_ARG;
  jrlqp_blockgi * s = new jrlqp_blockgi();
  *out = s;
  s->device = device;
  s->capacity = batch_capacity;
  int rc = jrlqp_structured_create(&s->g, G, batch_capacity, device);
  if(rc != JRLQP_OK)
  {
    s->err = s->g ? s->g->err : "invalid structure of G";
    return rc;
  }
  s->n = s->g->n;
  if(s->n > 1024)
  {
    // the passes over Q hold entries tid + 128 j, j < 8, of a reflector and of the vector: entries past 1023 would never be
    // updated (blockgi_kernel<8>, blockgi.cuh)
    s->err = "n = " + std::to_string(s->n) + " exceeds 1024, the largest size the structured solver supports";
    return JRLQP_ERR_ARG;
  }
  s->cb = C->nblocks;
  int nv = 0, nc = 0;
  for(int i = 0; i < s->cb; ++i)
  {
    const int ni = C->nvar[i], mi = C->ncstr[i];
    if(ni < 1 || mi < 0 || C->ld[i] < ni || C->offset[i] < 0)
    {
      s->err = "invalid block of C (rows >= 1, columns >= 0, ld >= rows)";
      return JRLQP_ERR_ARG;
    }
    s->cnvar.push_back(ni);
    s->cncstr.push_back(mi);
    s->cld.push_back(C->ld[i]);
    s->coff.push_back(C->offset[i]);
    s->cvar0.push_back(nv);
    s->ccstr0.push_back(nc);
    for(int k = 0; k < mi; ++k) s->toblock.push_back(i);
    if(mi > 0) s->c_min_stride = std::max<long long>(s->c_min_stride, C->offset[i] + (long long)(mi - 1) * C->ld[i] + ni);
    nv += ni;
    nc += mi;
  }
  s->cvar0.push_back(nv);
  s->ccstr0.push_back(nc);
  if(s->cb > 0 && nv != s->n)
  {
    s->err = "the blocks of C do not cover the variables of G";
    return JRLQP_ERR_ARG;
  }
  s->mc = nc;
  s->nb = use_bounds ? s->n : 0;
  SCK(cudaSetDevice(device));
  SCK(upload(s->d_cnvar, s->cnvar));
  SCK(upload(s->d_cld, s->cld));
  SCK(upload(s->d_cvar0, s->cvar0));
  SCK(upload(s->d_ccstr0, s->ccstr0));
  SCK(upload(s->d_toblock, s->toblock));
  SCK(upload(s->d_coff, s->coff));
  SCK(cudaMalloc(&s->d_ticket, sizeof(unsigned long long)));
  SCK(cudaMalloc(&s->d_gshared, sizeof(double) * std::max<long long>(1, s->g->min_stride)));
  SCK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  return configure(s);
}

int jrlqp_blockgi_destroy(jrlqp_blockgi * s)
{
  if(!s) return JRLQP_OK;
  cudaSetDevice(s->device);
  void * ptrs[] = {s->d_cnvar, s->d_cld, s->d_cvar0, s->d_ccstr0, s->d_toblock, s->d_coff, s->d_ws, s->d_ticket, s->d_ok, s->d_gshared, s->d_in, s->d_out};
  for(void * p : ptrs)
    if(p) cudaFree(p);
  if(s->stream) cudaStreamDestroy(s->stream);
  if(s->g) jrlqp_structured_destroy(s->g);
  delete s;
  return JRLQP_OK;
}

const char * jrlqp_blockgi_last_error(const jrlqp_blockgi * s)
{
  return s ? s->err.c_str() : "null handle";
}

int jrlqp_blockgi_set_options(jrlqp_blockgi * s, const jrlqp_options * o)
{
  if(!s || !o || o->max_iter < 0) return JRLQP_ERR_ARG;
  s->opt = *o;
  SCK(cudaSetDevice(s->device));
  return configure(s);
}

int jrlqp_blockgi_get_options(const jrlqp_blockgi * s, jrlqp_options * o)
{
  if(!s || !o) return JRLQP_ERR_ARG;
  *o = s->opt;
  return JRLQP_OK;
}

int jrlqp_blockgi_get_info(const jrlqp_blockgi * s, jrlqp_blockgi_info * info)
{
  if(!s || !info) return JRLQP_ERR_ARG;
  info->n = s->n;
  info->mc = s->mc;
  info->nb = s->nb;
  info->threads = s->bthreads ? s->bthreads : s->g->threads;
  info->smem_bytes = s->smem;
  info->ctas_per_sm = s->occ;
  info->grid = s->grid;
  info->num_sms = s->g->num_sms;
  info->workspace_bytes_per_cta = s->ws_stride * 8;
  info->g_elements_per_instance = s->g->touched;
  return JRLQP_OK;
}

int jrlqp_blockgi_solve_device(jrlqp_blockgi * s, const jrlqp_block_problem * pb, const jrlqp_result * res, void * stream_)
{
  if(!s || !pb || !res || pb->batch < 0) return JRLQP_ERR_ARG;
  if(!pb->G || !pb->a || !res->x) return JRLQP_ERR_ARG;
  if(s->mc > 0 && (!pb->C || !pb->bl || !pb->bu)) return JRLQP_ERR_ARG;
  if(s->nb > 0 && (!pb->xl || !pb->xu)) return JRLQP_ERR_ARG;
  if(pb->G_stride != 0 && pb->batch > 1 && pb->G_stride < s->g->min_stride) return JRLQP_ERR_ARG;
  if(pb->C_stride != 0 && pb->batch > 1 && pb->C_stride < s->c_min_stride) return JRLQP_ERR_ARG;
  if(pb->batch == 0) return JRLQP_OK;
  cudaStream_t stream = (cudaStream_t)stream_;
  SCK(cudaSetDevice(s->device));
  int rc = configure(s);
  if(rc != JRLQP_OK) return rc;
  const bool shared = pb->G_stride == 0;
  const long long nllt = shared ? 1 : pb->batch;
  if(nllt > s->ok_cap)
  {
    if(s->d_ok) cudaFree(s->d_ok);
    s->d_ok = nullptr;
    s->ok_cap = 0;
    SCK(cudaMalloc(&s->d_ok, sizeof(int) * nllt));
    s->ok_cap = nllt;
  }
  // pb_.G.lltInPlace() (src/experimental/BlockGISolver.cpp:71): in place on the caller's blocks; a shared G is
  // factorised once, in a private copy (every instance would compute the same factor)
  double * gdata = pb->G;
  if(shared)
  {
    SCK(cudaMemcpyAsync(s->d_gshared, pb->G, sizeof(double) * s->g->min_stride, cudaMemcpyDeviceToDevice, stream));
    gdata = s->d_gshared;
  }
  rc = jrlqp_structured_llt_device(s->g, gdata, shared ? s->g->min_stride : pb->G_stride, nllt, s->d_ok, stream);
  if(rc != JRLQP_OK)
  {
    s->err = s->g->err;
    return rc;
  }
  SCK(cudaMemsetAsync(s->d_ticket, 0, sizeof(unsigned long long), stream));
  BlockGiParams p{};
  p.G = base_params(s->g);
  p.G.data = gdata;
  p.G.stride = shared ? 0 : pb->G_stride;
  p.G.batch = pb->batch;
  p.llt_ok = s->d_ok;
  p.ok_stride = shared ? 0 : 1;
  p.cb = s->cb;
  p.cnvar = s->d_cnvar;
  p.coff = s->d_coff;
  p.cld = s->d_cld;
  p.cvar0 = s->d_cvar0;
  p.ccstr0 = s->d_ccstr0;
  p.toblock = s->d_toblock;
  p.mc = s->mc;
  p.nb = s->nb;
  p.max_iter = s->opt.max_iter;
  p.big_bnd = s->opt.big_bnd;
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
  p.x = res->x;
  p.u = res->u;
  p.f = res->f;
  p.iters = res->iterations;
  p.status = res->status;
  p.act = reinterpret_cast<signed char *>(res->active_set);
  p.alist = res->active_list;
  p.nact = res->n_active;
  p.qdoubles = nullptr;
  p.ws = s->d_ws;
  p.ws_stride = s->ws_stride;
  p.qcap = s->qcap;
  p.batch = pb->batch;
  p.ticket = s->d_ticket;
  // the warp-level solves stream the tiles by bulk copies: 16-byte aligned instances (the offsets inside one are even)
  const bool aligned = (reinterpret_cast<uintptr_t>(gdata) % 16) == 0 && (p.G.stride % 2) == 0;
  p.fast_nb = aligned ? s->fast_nb : 0;
  p.flags = s->flags;
  const long long grid = std::min<long long>(pb->batch, s->grid);
  s->kernel<<<(unsigned)grid, s->bthreads, s->smem, stream>>>(p);
  count_launch();
  SCK(cudaGetLastError());
  return JRLQP_OK;
}

int jrlqp_blockgi_solve_host(jrlqp_blockgi * s, const jrlqp_block_problem * pb, const jrlqp_result * res)
{
  if(!s || !pb || !res || pb->batch < 0) return JRLQP_ERR_ARG;
  if(!pb->G || !pb->a || !res->x) return JRLQP_ERR_ARG;
  if(pb->batch > s->capacity) return JRLQP_ERR_CAPACITY;
  if(pb->batch == 0) return 0;
  SCK(cudaSetDevice(s->device));
  const long long B = pb->batch;
  const int n = s->n, mc = s->mc, nb = s->nb, m = mc + nb;
  // input staging: every array takes B * stride elements (or one instance when shared)
  struct In
  {
    const double * h;
    long long stride, one;
    long long off;
  };
  In in[7] = {{pb->G, pb->G_stride, s->g->min_stride, 0}, {pb->a, pb->a_stride, n, 0},     {mc ? pb->C : nullptr, pb->C_stride, s->c_min_stride, 0},
              {mc ? pb->bl : nullptr, pb->bl_stride, mc, 0}, {mc ? pb->bu : nullptr, pb->bu_stride, mc, 0}, {nb ? pb->xl : nullptr, pb->xl_stride, n, 0},
              {nb ? pb->xu : nullptr, pb->xu_stride, n, 0}};
  long long tot = 0;
  for(auto & e : in)
  {
    if(!e.h) continue;
    if(e.stride != 0 && e.stride < e.one && B > 1) return JRLQP_ERR_ARG;
    e.off = tot;
    tot += ((e.stride == 0 ? e.one : (B - 1) * e.stride + e.one) + 1) & ~1LL;
  }
  if(tot * 8 > s->d_in_bytes)
  {
    if(s->d_in) cudaFree(s->d_in);
    s->d_in = nullptr;
    s->d_in_bytes = 0;
    SCK(cudaMalloc(&s->d_in, tot * 8));
    s->d_in_bytes = tot * 8;
  }
  // outputs: x, u, f (doubles), iterations, status, n_active, active_list (ints), active_set (bytes)
  const long long o_x = 0, o_u = o_x + B * n, o_f = o_u + B * m, nd = o_f + B;
  const long long o_it = 0, o_st = o_it + B, o_na = o_st + B, o_al = o_na + B, ni = o_al + B * n;
  const long long out_bytes = nd * 8 + ni * 4 + B * m;
  if(out_bytes > s->d_out_bytes)
  {
    if(s->d_out) cudaFree(s->d_out);
    s->d_out = nullptr;
    s->d_out_bytes = 0;
    SCK(cudaMalloc(&s->d_out, out_bytes));
    s->d_out_bytes = out_bytes;
  }
  double * od = reinterpret_cast<double *>(s->d_out);
  int * oi = reinterpret_cast<int *>(s->d_out + nd * 8);
  signed char * ob = reinterpret_cast<signed char *>(s->d_out + nd * 8 + ni * 4);
  for(auto & e : in)
  {
    if(!e.h) continue;
    const long long cnt = e.stride == 0 ? e.one : (B - 1) * e.stride + e.one;
    SCK(cudaMemcpyAsync(s->d_in + e.off, e.h, sizeof(double) * cnt, cudaMemcpyHostToDevice, s->stream));
  }
  jrlqp_block_problem dp = *pb;
  dp.G = s->d_in + in[0].off;
  dp.a = s->d_in + in[1].off;
  dp.C = mc ? s->d_in + in[2].off : nullptr;
  dp.bl = mc ? s->d_in + in[3].off : nullptr;
  dp.bu = mc ? s->d_in + in[4].off : nullptr;
  dp.xl = nb ? s->d_in + in[5].off : nullptr;
  dp.xu = nb ? s->d_in + in[6].off : nullptr;
  jrlqp_result dr{};
  dr.x = od + o_x;
  dr.u = od + o_u;
  dr.f = od + o_f;
  dr.iterations = oi + o_it;
  dr.status = oi + o_st;
  dr.n_active = oi + o_na;
  dr.active_list = oi + o_al;
  dr.active_set = reinterpret_cast<int8_t *>(ob);
  int rc = jrlqp_blockgi_solve_device(s, &dp, &dr, s->stream);
  if(rc != JRLQP_OK) return rc;
  std::vector<int> hst((size_t)B);
  SCK(cudaMemcpyAsync(res->x, dr.x, sizeof(double) * B * n, cudaMemcpyDeviceToHost, s->stream));
  if(res->u) SCK(cudaMemcpyAsync(res->u, dr.u, sizeof(double) * B * m, cudaMemcpyDeviceToHost, s->stream));
  if(res->f) SCK(cudaMemcpyAsync(res->f, dr.f, sizeof(double) * B, cudaMemcpyDeviceToHost, s->stream));
  if(res->iterations) SCK(cudaMemcpyAsync(res->iterations, dr.iterations, sizeof(int) * B, cudaMemcpyDeviceToHost, s->stream));
  SCK(cudaMemcpyAsync(hst.data(), dr.status, sizeof(int) * B, cudaMemcpyDeviceToHost, s->stream));
  if(res->n_active) SCK(cudaMemcpyAsync(res->n_active, dr.n_active, sizeof(int) * B, cudaMemcpyDeviceToHost, s->stream));
  if(res->active_list) SCK(cudaMemcpyAsync(res->active_list, dr.active_list, sizeof(int) * B * n, cudaMemcpyDeviceToHost, s->stream));
  if(res->active_set) SCK(cudaMemcpyAsync(res->active_set, dr.active_set, (size_t)(B * m), cudaMemcpyDeviceToHost, s->stream));
  SCK(cudaStreamSynchronize(s->stream));
  int worst = 0;
  for(long long k = 0; k < B; ++k)
  {
    if(res->status) res->status[k] = hst[(size_t)k];
    worst = std::max(worst, hst[(size_t)k]);
  }
  return worst;
}

} // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// Test harness of the orthonormal sequence (include/jrlqp_b200.h: jrlqp_blockgi_test_sequence)
// ---------------------------------------------------------------------------------------------------------------
extern "C" int jrlqp_blockgi_test_sequence(int32_t device, int32_t n, int32_t nrec, const int32_t * rec, const double * qdata, int64_t qlen,
                                           double * v, int32_t ncases, int32_t transpose, int32_t threads)
{
  if(n < 2 || nrec < 0 || !rec || !qdata || !v || ncases < 1 || threads < 128 || threads % 32 != 0 || threads > 1024 || n > 1024) return JRLQP_ERR_ARG;
  if(cudaSetDevice(device) != cudaSuccess) return JRLQP_ERR_CUDA;
  const long long rsz = (long long)n * (n + 1) / 2;
  double *d_ws = nullptr, *d_v = nullptr;
  int * d_rec = nullptr;
  bool ok = cudaMalloc(&d_ws, sizeof(double) * (rsz + qlen + 1)) == cudaSuccess && cudaMalloc(&d_v, sizeof(double) * (size_t)n * ncases) == cudaSuccess &&
            cudaMalloc(&d_rec, sizeof(int) * (3 * (size_t)nrec + 1)) == cudaSuccess;
  ok = ok && cudaMemcpy(d_ws + rsz, qdata, sizeof(double) * qlen, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(d_v, v, sizeof(double) * (size_t)n * ncases, cudaMemcpyHostToDevice) == cudaSuccess;
  ok = ok && cudaMemcpy(d_rec, rec, sizeof(int) * 3 * (size_t)nrec, cudaMemcpyHostToDevice) == cudaSuccess;
  int rc = JRLQP_ERR_CUDA;
  if(ok)
  {
    BlockGiParams p{};
    p.G.n = n;
    p.G.nmax = 1;
    p.G.type = SG_TRI;
    p.mc = 0;
    p.nb = 0;
    p.max_iter = std::max(nrec, 1);
    p.ws = d_ws;
    p.ws_stride = 0;
    p.qcap = qlen;
    p.flags = 7;
    if(const char * e = getenv("JRLQP_BLOCKGI_FAST")) p.flags = atoi(e) & 7;
    const int smem = (int)BlockGi<8>::smem_bytes(n, 1, 0, p.max_iter, 0, 0);
    ok = jrlqp::raise_smem_limit(blockgi_sequence_test_kernel, smem) == cudaSuccess;
    if(ok)
    {
      blockgi_sequence_test_kernel<<<1, threads, smem>>>(p, d_rec, nrec, d_v, ncases, transpose);
      count_launch();
      ok = cudaDeviceSynchronize() == cudaSuccess && cudaMemcpy(v, d_v, sizeof(double) * (size_t)n * ncases, cudaMemcpyDeviceToHost) == cudaSuccess;
    }
    rc = ok ? JRLQP_OK : JRLQP_ERR_CUDA;
  }
  cudaFree(d_ws);
  cudaFree(d_v);
  cudaFree(d_rec);
  return rc;
}

#ifdef JRLQP_TEST_FALLBACKS
// test build only: this unit's fallback counters and decline flag (test_fallbacks.cuh), read and set through capi.cu
namespace jrlqp
{
int fb_collect_blockgi(unsigned long long * out) { return fb_collect(out); }
int fb_set_decline_blockgi(int on) { return fb_set_decline(on); }
} // namespace jrlqp
#endif
