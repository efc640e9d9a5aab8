// Host side of the structured-decomposition C-ABI (include/jrlqp_b200.h, jrlqp_structured_*):
// descriptor upload, launch configuration, and the host-pointer entry points. Pure CUDA runtime.
#include "smem_limit.hpp"
#include "structured_host.hpp"
#include "structured_small.cuh"

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <atomic>
#include <string>
#include <vector>

using namespace jrlqp;

namespace jrlqp
{
void count_launch(); // capi.cu: feeds jrlqp_launch_count()
}

namespace jrlqp
{

// ---------------------------------------------------------------------------------------------
// StructuredG::lltInPlace. Shared memory: 3 tiles of nmax x nmax + nmax doubles of scratch.
//   tri:   T0 = D_i (current), T1 = S_i, T2 = D_{i+1} (receives the rank update, becomes current)
//   arrow: T0 = D_i,           T1 = B_i, T2 = D_last  (resident, receives every rank update)
// ---------------------------------------------------------------------------------------------
__global__ void structured_llt_kernel(const StructParams P)
{
  extern __shared__ __align__(16) double sm[];
  const int tile = P.nmax * P.nmax;
  const int b = P.b;
  const bool tri = P.type == SG_TRI;
  const bool up = P.type == SG_ARROW_UP;
  for(long long inst = blockIdx.x; inst < P.batch; inst += gridDim.x)
  {
    double * base = P.data + inst * P.stride;
    double * cur = sm;
    double * S = sm + tile;
    double * nxt = sm + 2 * tile;
    double * vd = sm + 3 * tile;
    bool ok = true;
    const int last = up ? 0 : b - 1; // block that ends the permuted system
    if(tri)
      load_tile(cur, base + P.doff[0], P.size[0], P.size[0], P.dld[0], false);
    else
      load_tile(nxt, base + P.doff[last], P.size[last], P.size[last], P.dld[last], false);
    for(int i = 0; i < b - 1 && ok; ++i)
    {
      const int di = tri ? i : (up ? i + 1 : i); // get<Up>::D(diag, i)
      const int ni = P.size[di];
      // off-diagonal block i as stored: tri n_{i+1} x n_i, down n_last x n_i, up n_{i+1} x n_0 (= B_i^T)
      const int srows = tri ? P.size[i + 1] : (up ? P.size[i + 1] : P.size[last]);
      const int scols = up ? P.size[0] : ni;
      const int brows = up ? scols : srows; // rows of B_i once in shared memory (B_i: brows x ni)
      if(!tri) load_tile(cur, base + P.doff[di], ni, ni, P.dld[di], false);
      load_tile(S, base + P.ooff[i], srows, scols, P.old[i], up);
      if(tri) load_tile(nxt, base + P.doff[i + 1], srows, srows, P.dld[i + 1], false);
      __syncthreads();
      ok = tile_chol(cur, ni, vd); // Li = chol(Di)
      if(ok)
      {
        tile_trsm_right_lt(S, brows, cur, ni); // Bi = Bi Li^-T
        __syncthreads();
        tile_syrk_sub(nxt, brows, S, ni); // D_{i+1} (tri) or D_last (arrow) -= Bi Bi^T
        store_tile(base + P.doff[di], cur, ni, ni, P.dld[di], false, true);
        store_tile(base + P.ooff[i], S, srows, scols, P.old[i], up, false);
      }
      __syncthreads();
      if(tri)
      {
        double * t = cur;
        cur = nxt;
        nxt = t;
      }
    }
    if(ok)
    {
      double * Dl = tri ? cur : nxt;
      const int nl = P.size[last];
      __syncthreads();
      ok = tile_chol(Dl, nl, vd);
      if(ok) store_tile(base + P.doff[last], Dl, nl, nl, P.dld[last], false, true);
    }
    if(threadIdx.x == 0 && P.ok) P.ok[inst] = ok ? 1 : 0;
    __syncthreads();
  }
}

// StructuredG::solveL / solveInPlaceLTranspose with the reference's start / end hints.
// Shared memory: v[n] (the right-hand side / solution), then 2 tiles of nmax x nmax (L_i, B_i).
__global__ void structured_solve_kernel(const StructParams P)
{
  extern __shared__ __align__(16) double sm[];
  const int n = P.n;
  double * v = sm;
  double * Lt = sm + ((n + 1) & ~1);
  double * Bt = Lt + P.nmax * P.nmax;
  const bool up = P.type == SG_ARROW_UP;
  const long long work = P.batch * P.ncols;
  for(long long w = blockIdx.x; w < work; w += gridDim.x)
  {
    const long long inst = w / P.ncols;
    const int col = (int)(w - inst * P.ncols);
    const double * base = P.data + inst * P.stride;
    double * Mc = P.M + inst * P.mstride + (long long)col * P.ldm;

    // load the column (up arrow, L solve: v = P^T m, src/decomposition/blockArrowLLT.cpp:163-169)
    const bool perm_in = up && !P.transpose;
    for(int i = threadIdx.x; i < n; i += blockDim.x) v[perm_in ? sg_perm(P, i) : i] = Mc[i];
    __syncthreads();
    sg_solve_inplace(P, base, v, Lt, Bt, P.transpose != 0, P.hint_start, P.hint_end);
    // store (up arrow, L^T solve: m = P v, src/decomposition/blockArrowLLT.cpp:264-270)
    const bool perm_out = up && P.transpose;
    for(int i = threadIdx.x; i < n; i += blockDim.x) Mc[i] = v[perm_out ? sg_perm(P, i) : i];
    __syncthreads();
  }
}

} // namespace jrlqp

namespace
{

void off_shape(const jrlqp_structured * s, int i, int & rows, int & cols)
{
  if(s->type == SG_TRI)
  {
    rows = s->size[i + 1];
    cols = s->size[i];
  }
  else if(s->type == SG_ARROW_DOWN)
  {
    rows = s->size[s->b - 1];
    cols = s->size[i];
  }
  else
  {
    rows = s->size[i + 1];
    cols = s->size[0];
  }
}

} // namespace

extern "C"
{

int jrlqp_structured_create(jrlqp_structured ** out, const jrlqp_structure * st, int64_t batch_capacity, int32_t device)
{
  if(!out) return JRLQP_ERR_ARG;
  *out = nullptr;
  if(!st || st->nblocks < 1 || st->type < 0 || st->type > 2 || batch_capacity < 0) return JRLQP_ERR_ARG;
  if(!st->block_size || !st->diag_offset || !st->diag_ld) return JRLQP_ERR_ARG;
  if(st->nblocks > 1 && (!st->off_offset || !st->off_ld)) return JRLQP_ERR_ARG;
  jrlqp_structured * s = new jrlqp_structured();
  *out = s;
  s->type = st->type;
  s->b = st->nblocks;
  s->capacity = batch_capacity;
  s->device = device;
  s->start.push_back(0);
  for(int i = 0; i < s->b; ++i)
  {
    const int ni = st->block_size[i];
    if(ni < 1 || ni > 96 || st->diag_ld[i] < ni || st->diag_offset[i] < 0)
    {
      s->err = "invalid diagonal block (size must be in [1, 96], ld >= size)";
      return JRLQP_ERR_ARG;
    }
    s->size.push_back(ni);
    s->doff.push_back(st->diag_offset[i]);
    s->dld.push_back(st->diag_ld[i]);
    s->n += ni;
    s->start.push_back(s->n);
    s->nmax = std::max(s->nmax, ni);
    s->min_stride = std::max<long long>(s->min_stride, st->diag_offset[i] + (long long)(ni - 1) * st->diag_ld[i] + ni);
    s->touched += (long long)ni * (ni + 1) / 2;
  }
  for(int i = 0; i + 1 < s->b; ++i)
  {
    int rows, cols;
    off_shape(s, i, rows, cols);
    if(st->off_ld[i] < rows || st->off_offset[i] < 0)
    {
      s->err = "invalid off-diagonal block (ld < rows)";
      return JRLQP_ERR_ARG;
    }
    s->ooff.push_back(st->off_offset[i]);
    s->old.push_back(st->off_ld[i]);
    s->min_stride = std::max<long long>(s->min_stride, st->off_offset[i] + (long long)(cols - 1) * st->off_ld[i] + rows);
    s->touched += (long long)rows * cols;
  }
  int ndev = 0;
  SCK(cudaGetDeviceCount(&ndev));
  if(device < 0 || device >= ndev)
  {
    s->err = "no such CUDA device";
    return JRLQP_ERR_CUDA;
  }
  SCK(cudaSetDevice(device));
  cudaDeviceProp prop;
  SCK(cudaGetDeviceProperties(&prop, device));
  if(prop.major != 10)
  {
    s->err = "this library contains sm_100a code only (Blackwell B200 required)";
    return JRLQP_ERR_CUDA;
  }
  s->num_sms = prop.multiProcessorCount;
  s->threads = s->nmax <= 32 ? 32 : (s->nmax <= 64 ? 64 : 128);
  const int tile = s->nmax * s->nmax;
  s->llt_smem = (3 * tile + s->nmax + 2) * 8;
  s->solve_smem = (((s->n + 1) & ~1) + 2 * tile) * 8;
  if(std::max(s->llt_smem, s->solve_smem) > (int)prop.sharedMemPerBlockOptin)
  {
    s->err = "structure does not fit in shared memory";
    return JRLQP_ERR_ARG;
  }
  SCK(jrlqp::raise_smem_limit(structured_llt_kernel, s->llt_smem));
  SCK(jrlqp::raise_smem_limit(structured_solve_kernel, s->solve_smem));
  SCK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s->llt_occ, structured_llt_kernel, s->threads, s->llt_smem));
  SCK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s->solve_occ, structured_solve_kernel, s->threads, s->solve_smem));
  if(s->llt_occ < 1 || s->solve_occ < 1)
  {
    s->err = "kernel cannot be made resident";
    return JRLQP_ERR_ARG;
  }
  SCK(upload(s->d_size, s->size));
  SCK(upload(s->d_dld, s->dld));
  SCK(upload(s->d_old, s->old));
  SCK(upload(s->d_start, s->start));
  SCK(upload(s->d_doff, s->doff));
  SCK(upload(s->d_ooff, s->ooff));
  SCK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  // eligibility for the small-tile kernel
  {
    const int nb = s->size[0];
    bool okk = s->type == SG_TRI && (nb == 8 || nb == 12 || nb == 16);
    for(int i = 0; i < s->b && okk; ++i) okk = s->size[i] == nb && s->dld[i] == nb && (s->doff[i] % 2) == 0;
    for(int i = 0; i + 1 < s->b && okk; ++i) okk = s->old[i] == nb && (s->ooff[i] % 2) == 0;
    s->small_nb = okk ? nb : 0;
    if(const char * e = getenv("JRLQP_STRUCT_KERNEL")) s->kernel_mode = atoi(e);
  }
  return JRLQP_OK;
}

int jrlqp_structured_set_kernel(jrlqp_structured * s, int32_t mode)
{
  if(!s || mode < 0 || mode > 3) return JRLQP_ERR_ARG;
  if(mode >= 2 && s->small_nb == 0)
  {
    s->err = "the small-tile kernel needs a tri-block-diagonal chain of uniform dense tiles of 8, 12 or 16 rows";
    return JRLQP_ERR_ARG;
  }
  s->kernel_mode = mode;
  return JRLQP_OK;
}

int jrlqp_structured_destroy(jrlqp_structured * s)
{
  if(!s) return JRLQP_OK;
  cudaSetDevice(s->device);
  void * ptrs[] = {s->d_size, s->d_dld, s->d_old, s->d_start, s->d_doff, s->d_ooff, s->d_data, s->d_M, s->d_ok};
  for(void * p : ptrs)
    if(p) cudaFree(p);
  if(s->stream) cudaStreamDestroy(s->stream);
  delete s;
  return JRLQP_OK;
}

const char * jrlqp_structured_last_error(const jrlqp_structured * s)
{
  return s ? s->err.c_str() : "null handle";
}

int jrlqp_structured_get_info(const jrlqp_structured * s, jrlqp_structured_info * info)
{
  if(!s || !info) return JRLQP_ERR_ARG;
  info->threads = s->threads;
  info->llt_smem_bytes = s->llt_smem;
  info->llt_ctas_per_sm = s->llt_occ;
  info->solve_smem_bytes = s->solve_smem;
  info->solve_ctas_per_sm = s->solve_occ;
  info->num_sms = s->num_sms;
  info->elements_per_instance = s->touched;
  return JRLQP_OK;
}

int jrlqp_structured_llt_device(jrlqp_structured * s, double * data, int64_t stride, int64_t batch, int32_t * ok, void * stream)
{
  if(!s || !data || batch < 0) return JRLQP_ERR_ARG;
  if(batch > 1 && stride < s->min_stride) return JRLQP_ERR_ARG; // instances would overlap
  if(batch == 0) return JRLQP_OK;
  SCK(cudaSetDevice(s->device));
  StructParams p = base_params(s);
  p.data = data;
  p.stride = stride;
  p.batch = batch;
  p.ok = ok;
  // small uniform tiles: two instances per warp, tiles in registers (structured_small.cuh); needs 16-byte aligned instances
  const bool aligned = (reinterpret_cast<uintptr_t>(data) % 16) == 0 && (stride % 2) == 0;
  constexpr int kDefaultSmall = 3; // automatic mode on an eligible structure: 2 = small tiles (plain loads), 3 = small tiles + TMA
  const int mode = s->kernel_mode == 0 ? (s->small_nb && aligned ? kDefaultSmall : 1) : s->kernel_mode;
  if(mode >= 2 && s->small_nb && aligned)
  {
    const bool tma = mode == 3;
    const int nb = s->small_nb, tt = nb * nb;
    const int smem = 4 * (2 * tt + (tma ? 8 * tt + 2 : 0)) * 8;
    void (*fn)(const StructParams) = nullptr;
    if(nb == 8) fn = tma ? structured_llt_small_kernel<8, true> : structured_llt_small_kernel<8, false>;
    if(nb == 12) fn = tma ? structured_llt_small_kernel<12, true> : structured_llt_small_kernel<12, false>;
    if(nb == 16) fn = tma ? structured_llt_small_kernel<16, true> : structured_llt_small_kernel<16, false>;
    SCK(jrlqp::raise_smem_limit(fn, smem));
    int occ = 0;
    SCK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 128, smem));
    const long long pairs = (batch + 1) / 2;
    const long long grid = std::min<long long>((pairs + 3) / 4, (long long)std::max(occ, 1) * s->num_sms);
    fn<<<(unsigned)grid, 128, smem, (cudaStream_t)stream>>>(p);
    count_launch();
    SCK(cudaGetLastError());
    return JRLQP_OK;
  }
  const long long grid = std::min<long long>(batch, (long long)s->llt_occ * s->num_sms);
  structured_llt_kernel<<<(unsigned)grid, s->threads, s->llt_smem, (cudaStream_t)stream>>>(p);
  count_launch();
  SCK(cudaGetLastError());
  return JRLQP_OK;
}

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
                                  void * stream)
{
  if(!s || !data || !M || batch < 0 || ncols < 0 || ldm < s->n) return JRLQP_ERR_ARG;
  if(start < 0 || start > s->n || end > s->n) return JRLQP_ERR_ARG;
  if(batch == 0 || ncols == 0) return JRLQP_OK;
  SCK(cudaSetDevice(s->device));
  StructParams p = base_params(s);
  p.data = const_cast<double *>(data);
  p.stride = stride;
  p.batch = batch;
  p.M = M;
  p.ldm = ldm;
  p.ncols = ncols;
  p.mstride = m_stride;
  p.transpose = transpose ? 1 : 0;
  p.hint_start = start;
  p.hint_end = end;
  // small uniform tiles: one column per warp, solved in place, tiles streamed by TMA (structured_small.cuh); needs 16-byte
  // aligned instances (the offsets inside one are even)
  const bool aligned = (reinterpret_cast<uintptr_t>(data) % 16) == 0 && (stride % 2) == 0;
  const int mode = s->kernel_mode == 0 ? (s->small_nb && aligned ? 3 : 1) : s->kernel_mode;
  if(mode >= 2 && s->small_nb && aligned)
  {
    const int nb = s->small_nb;
    void (*fn)(const StructParams) = nb == 8 ? structured_solve_small_kernel<8> : (nb == 12 ? structured_solve_small_kernel<12> : structured_solve_small_kernel<16>);
    const long long per_warp = TriWarp::ring_doubles(nb) + TriWarp::RING + (TriWarp::RING & 1);
    const int smem = (int)((2LL * s->b + 4 * per_warp) * 8);
    SCK(jrlqp::raise_smem_limit(fn, smem));
    int occ = 0;
    SCK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 128, smem));
    if(occ >= 1)
    {
      const long long work = batch * ncols;
      const long long grid = std::min<long long>((work + 3) / 4, (long long)occ * s->num_sms);
      fn<<<(unsigned)grid, 128, smem, (cudaStream_t)stream>>>(p);
      count_launch();
      SCK(cudaGetLastError());
      return JRLQP_OK;
    }
  }
  const long long grid = std::min<long long>(batch * ncols, (long long)s->solve_occ * s->num_sms);
  structured_solve_kernel<<<(unsigned)grid, s->threads, s->solve_smem, (cudaStream_t)stream>>>(p);
  count_launch();
  SCK(cudaGetLastError());
  return JRLQP_OK;
}

static int ensure_data(jrlqp_structured * s, long long elems)
{
  if(elems > s->d_data_elems)
  {
    if(s->d_data) cudaFree(s->d_data);
    s->d_data = nullptr;
    s->d_data_elems = 0;
    SCK(cudaMalloc(&s->d_data, sizeof(double) * elems));
    s->d_data_elems = elems;
  }
  if(!s->d_ok) SCK(cudaMalloc(&s->d_ok, sizeof(int) * std::max<long long>(s->capacity, 1)));
  return JRLQP_OK;
}

int jrlqp_structured_llt_host(jrlqp_structured * s, double * data, int64_t stride, int64_t batch, int32_t * ok)
{
  if(!s || !data || batch < 0) return JRLQP_ERR_ARG;
  if(batch > s->capacity) return JRLQP_ERR_CAPACITY;
  if(batch == 0) return 0;
  if(stride < s->min_stride) return JRLQP_ERR_ARG;
  SCK(cudaSetDevice(s->device));
  const long long elems = (long long)batch * stride;
  int rc = ensure_data(s, elems);
  if(rc != JRLQP_OK) return rc;
  SCK(cudaMemcpyAsync(s->d_data, data, sizeof(double) * elems, cudaMemcpyHostToDevice, s->stream));
  rc = jrlqp_structured_llt_device(s, s->d_data, stride, batch, s->d_ok, s->stream);
  if(rc != JRLQP_OK) return rc;
  SCK(cudaMemcpyAsync(data, s->d_data, sizeof(double) * elems, cudaMemcpyDeviceToHost, s->stream));
  std::vector<int> hok((size_t)batch);
  SCK(cudaMemcpyAsync(hok.data(), s->d_ok, sizeof(int) * batch, cudaMemcpyDeviceToHost, s->stream));
  SCK(cudaStreamSynchronize(s->stream));
  int failed = 0;
  for(long long k = 0; k < batch; ++k)
  {
    if(ok) ok[k] = hok[(size_t)k];
    failed += hok[(size_t)k] ? 0 : 1;
  }
  return failed;
}

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
                                int32_t end)
{
  if(!s || !data || !M || batch < 0 || ncols < 0 || ldm < s->n) return JRLQP_ERR_ARG;
  if(batch > s->capacity) return JRLQP_ERR_CAPACITY;
  if(batch == 0 || ncols == 0) return JRLQP_OK;
  if(stride < s->min_stride || m_stride < (long long)(ncols - 1) * ldm + s->n) return JRLQP_ERR_ARG;
  SCK(cudaSetDevice(s->device));
  const long long elems = (long long)batch * stride;
  int rc = ensure_data(s, elems);
  if(rc != JRLQP_OK) return rc;
  const long long melems = (long long)batch * m_stride;
  if(melems > s->d_M_elems)
  {
    if(s->d_M) cudaFree(s->d_M);
    s->d_M = nullptr;
    s->d_M_elems = 0;
    SCK(cudaMalloc(&s->d_M, sizeof(double) * melems));
    s->d_M_elems = melems;
  }
  SCK(cudaMemcpyAsync(s->d_data, data, sizeof(double) * elems, cudaMemcpyHostToDevice, s->stream));
  SCK(cudaMemcpyAsync(s->d_M, M, sizeof(double) * melems, cudaMemcpyHostToDevice, s->stream));
  rc = jrlqp_structured_solve_device(s, s->d_data, stride, s->d_M, ldm, ncols, m_stride, batch, transpose, start, end, s->stream);
  if(rc != JRLQP_OK) return rc;
  SCK(cudaMemcpyAsync(M, s->d_M, sizeof(double) * melems, cudaMemcpyDeviceToHost, s->stream));
  SCK(cudaStreamSynchronize(s->stream));
  return JRLQP_OK;
}

} // extern "C"

#ifdef JRLQP_TEST_FALLBACKS
// test build only: this unit's fallback counters and decline flag (test_fallbacks.cuh), read and set through capi.cu
namespace jrlqp
{
int fb_collect_structured(unsigned long long * out) { return fb_collect(out); }
int fb_set_decline_structured(int on) { return fb_set_decline(on); }
} // namespace jrlqp
#endif
