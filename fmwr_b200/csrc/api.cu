// C ABI (include/fmwr_b200.h): context, model handles, link tables and the one-shot
// host-buffer entry points that stand behind FM() / FMPredict() / FMTrack()
// (reference src/FM.cpp:7, :177, :218).
#include "forward.cuh"

#include <chrono>
#include <cmath>
#include <exception>
#include <map>
#include <mutex>

namespace fmwr {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

// ---- caching device allocator -------------------------------------------------------------------------------
static std::mutex g_mem_mu;
static std::map<std::pair<int, size_t>, std::vector<void*>> g_mem_cache;   // (device, rounded bytes) -> free blocks

static size_t round_bytes(size_t b)
{
  const size_t g = b >= (8u << 20) ? (2u << 20) : 512u;      // 2 MiB granules for big blocks, 512 B for small ones
  return (b + g - 1) / g * g;
}

void dev_trim()
{
  std::lock_guard<std::mutex> lk(g_mem_mu);
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& kv : g_mem_cache) {
    if (kv.second.empty()) continue;
    cudaSetDevice(kv.first.first);
    for (void* p : kv.second) cudaFree(p);
    kv.second.clear();
  }
  cudaSetDevice(cur);
}

void* dev_alloc(size_t bytes)
{
  const size_t rb = round_bytes(bytes);
  int dev = 0;
  FMWR_CUDA(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lk(g_mem_mu);
    auto it = g_mem_cache.find({dev, rb});
    if (it != g_mem_cache.end() && !it->second.empty()) {
      void* p = it->second.back();
      it->second.pop_back();
      return p;
    }
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, rb);
  if (e == cudaErrorMemoryAllocation) {
    cudaGetLastError();
    dev_trim();
    e = cudaMalloc(&p, rb);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    char b[160];
    snprintf(b, sizeof b, "CUDA error %s allocating %zu bytes", cudaGetErrorString(e), rb);
    throw Error(e == cudaErrorMemoryAllocation ? FMWR_ERR_NOMEM : FMWR_ERR_CUDA, b);
  }
  return p;
}

void dev_free(void* p, size_t bytes)
{
  if (!p) return;
  // Normal paths synchronise their stream before a buffer goes out of scope.  While an exception unwinds, kernels that
  // reference the block may still be queued: wait for the device before the block can be handed to another stream / context.
  if (std::uncaught_exceptions() > 0) { cudaDeviceSynchronize(); cudaGetLastError(); }
  int dev = 0;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) == cudaSuccess) dev = attr.device; else { cudaGetLastError(); cudaGetDevice(&dev); }
  std::lock_guard<std::mutex> lk(g_mem_mu);
  g_mem_cache[{dev, round_bytes(bytes)}].push_back(p);
}

cudaEvent_t prof_begin(fmwr_ctx* ctx, const char* tag)
{
  cudaEvent_t e[2];
  for (int i = 0; i < 2; ++i) {
    if (!ctx->prof_pool.empty()) { e[i] = ctx->prof_pool.back(); ctx->prof_pool.pop_back(); }
    else if (cudaEventCreate(&e[i]) != cudaSuccess) return nullptr;
  }
  cudaEventRecord(e[0], ctx->stream);
  ctx->prof_recs.push_back({tag, e[0], e[1]});
  return e[1];
}

int padded_k(int k, int prec)
{
  const int vn = prec == FMWR_F64 ? 2 : 4;
  int units = (k + vn - 1) / vn;
  if (units < 1) units = 1;
  int u = 1;
  while (u < units) u <<= 1;
  if (u > 128) throw Error(FMWR_ERR_UNSUPPORTED, "factor.number too large for this build (max 512 fp32 / 256 fp64)");
  return u * vn;
}

// ---- link tables -------------------------------------------------------------------------------
// The reference ships two lookup tables (src/util/RandomData.h: Phi on a 1/549.9667 grid, 2861 pts;
// src/util/RandomData_.h: phi/(1-Phi) on a 2e-4 grid over [-3,5], 40001 pts).  They are regenerated
// here from their defining formulas in fp64 (tests pin them against the reference tables).
__global__ void fill_pn_table(double* __restrict__ Y, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = (double)i / 549.966731401936;
  Y[i] = 0.5 * erfc(-x * 0.70710678118654752440);
}

__global__ void fill_dp_table(double* __restrict__ Y, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = rint((-3.0 + 2e-4 * (double)i) * 1e4) / 1e4;
  const double tail = 0.5 * erfc(x * 0.70710678118654752440);
  Y[i] = exp(-0.5 * x * x) / 2.5066282746310002 / tail;
}

void build_link_tables(fmwr_ctx* ctx)
{
  ctx->pn_table.alloc(2862);
  ctx->dp_table.alloc(40002);
  FMWR_LAUNCH(ctx, fill_pn_table, ceil_div(2862, 256), 256, 0, ctx->pn_table.p, 2862);
  FMWR_LAUNCH(ctx, fill_dp_table, ceil_div(40002, 256), 256, 0, ctx->dp_table.p, 40002);
}

__global__ void link_eval_kernel(int which, int64_t n, const double* __restrict__ x, const double* __restrict__ pn,
                                 const double* __restrict__ dp, double* __restrict__ out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = which == 0 ? dev_fast_pnorm(pn, x[i]) : dev_fast_dpnorm(dp, x[i]);
}

void link_table_eval(fmwr_ctx* ctx, int which, int64_t n, const double* x, double* out)
{
  DBuf<double> dx, dout;
  dx.alloc(n); dout.alloc(n);
  FMWR_CUDA(cudaMemcpyAsync(dx.p, x, 8 * n, cudaMemcpyHostToDevice, ctx->stream));
  FMWR_LAUNCH(ctx, link_eval_kernel, ceil_div(n, 256), 256, 0, which, n, dx.p, ctx->pn_table.p, ctx->dp_table.p, dout.p);
  FMWR_CUDA(cudaMemcpyAsync(out, dout.p, 8 * n, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
}

// ---- model <-> host ------------------------------------------------------------------------------
template <class T>
__global__ void pack_v(const double* __restrict__ src /*[p][k]*/, T* __restrict__ dst /*[p][kp]*/, int64_t p, int k, int kp)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p * kp) return;
  const int f = (int)(i % kp);
  const int64_t j = i / kp;
  dst[i] = f < k ? T(src[j * k + f]) : T(0);
}

template <class T>
__global__ void unpack_v(const T* __restrict__ src /*[p][kp]*/, double* __restrict__ dst /*[p][k]*/, int64_t p, int k, int kp)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p * k) return;
  const int f = (int)(i % k);
  const int64_t j = i / k;
  dst[i] = (double)src[j * kp + f];
}

template <class T>
__global__ void cast_from_f64(const double* __restrict__ src, T* __restrict__ dst, int64_t n)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = T(src[i]);
}

template <class T>
__global__ void cast_to_f64(const T* __restrict__ src, double* __restrict__ dst, int64_t n)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (double)src[i];
}

void model_set_host(fmwr_model* m, double w0, const double* w, const double* v)
{
  fmwr_ctx* ctx = m->ctx;
  const int64_t p = m->p;
  ctx->h2d_bytes += 8 + 8 * p + 8 * p * (int64_t)m->k;
  FMWR_CUDA(cudaMemsetAsync(m->scal.p, 0, m->scal.bytes(), ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(m->scal.p, &w0, 8, cudaMemcpyHostToDevice, ctx->stream));
  DBuf<double> stage;
  const int64_t vk = p * (int64_t)(m->k > 0 ? m->k : 1);
  stage.alloc(std::max<int64_t>(p, vk));
  if (p > 0) {
    FMWR_CUDA(cudaMemcpyAsync(stage.p, w, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
    if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, cast_from_f64<double>, ceil_div(p, 256), 256, 0, stage.p, (double*)m->w.p, p);
    else FMWR_LAUNCH(ctx, cast_from_f64<float>, ceil_div(p, 256), 256, 0, stage.p, (float*)m->w.p, p);
    if (m->k > 0) {
      FMWR_CUDA(cudaMemcpyAsync(stage.p, v, 8 * p * m->k, cudaMemcpyHostToDevice, ctx->stream));
      if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, pack_v<double>, ceil_div(p * m->kp, 256), 256, 0, stage.p, (double*)m->v.p, p, m->k, m->kp);
      else FMWR_LAUNCH(ctx, pack_v<float>, ceil_div(p * m->kp, 256), 256, 0, stage.p, (float*)m->v.p, p, m->k, m->kp);
    } else {
      FMWR_CUDA(cudaMemsetAsync(m->v.p, 0, m->v.bytes(), ctx->stream));
    }
  }
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
}

double model_get_w0(fmwr_model* m)
{
  double w0 = 0;
  FMWR_CUDA(cudaMemcpyAsync(&w0, m->scal.p, 8, cudaMemcpyDeviceToHost, m->ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(m->ctx->stream));
  return w0;
}

void model_get_host(fmwr_model* m, double* w0, double* w, double* v)
{
  fmwr_ctx* ctx = m->ctx;
  const int64_t p = m->p;
  if (w0) *w0 = model_get_w0(m);
  DBuf<double> stage;
  const int64_t vk = p * (int64_t)(m->k > 0 ? m->k : 1);
  stage.alloc(std::max<int64_t>(p, vk));
  ctx->d2h_bytes += (w0 ? 8 : 0) + (w ? 8 * p : 0) + (v ? 8 * p * (int64_t)m->k : 0);
  if (p > 0 && w) {
    if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, cast_to_f64<double>, ceil_div(p, 256), 256, 0, (const double*)m->w.p, stage.p, p);
    else FMWR_LAUNCH(ctx, cast_to_f64<float>, ceil_div(p, 256), 256, 0, (const float*)m->w.p, stage.p, p);
    FMWR_CUDA(cudaMemcpyAsync(w, stage.p, 8 * p, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (p > 0 && v && m->k > 0) {
    if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, unpack_v<double>, ceil_div(p * m->k, 256), 256, 0, (const double*)m->v.p, stage.p, p, m->k, m->kp);
    else FMWR_LAUNCH(ctx, unpack_v<float>, ceil_div(p * m->k, 256), 256, 0, (const float*)m->v.p, stage.p, p, m->k, m->kp);
    FMWR_CUDA(cudaMemcpyAsync(v, stage.p, 8 * p * m->k, cudaMemcpyDeviceToHost, ctx->stream));
  }
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
}

// returns true when the existing state was kept (warm start)
bool model_alloc_state(fmwr_model* m, int n_state, int solver, bool warm)
{
  FMWR_REQUIRE(n_state <= 5, FMWR_ERR_ARG, "too many optimizer state arrays");
  bool have = m->n_state == n_state && m->state_solver == solver;
  for (int i = 0; i < n_state && have; ++i)
    have = m->sw[i].p && m->sv[i].p && m->sw[i].bytes() == (size_t)(m->p + 4) * m->esz() && m->sv[i].bytes() == (size_t)m->p * m->kp * m->esz();
  if (warm && have) return true;
  for (int i = 0; i < n_state; ++i) {
    m->sw[i].alloc((size_t)(m->p + 4) * m->esz());      // +4 elements: 16-byte-rounded staging reads (update_tma.cuh)
    m->sv[i].alloc((size_t)m->p * m->kp * m->esz());
    FMWR_CUDA(cudaMemsetAsync(m->sw[i].p, 0, m->sw[i].bytes(), m->ctx->stream));
    FMWR_CUDA(cudaMemsetAsync(m->sv[i].p, 0, m->sv[i].bytes(), m->ctx->stream));
  }
  for (int i = n_state; i < 5; ++i) { m->sw[i].release(); m->sv[i].release(); }
  FMWR_CUDA(cudaMemsetAsync((double*)m->scal.p + 1, 0, 7 * sizeof(double), m->ctx->stream));     // Learner::init(): restart at zero
  m->n_state = n_state;
  m->state_solver = solver;
  return false;
}

fmwr_data* data_create_f64(fmwr_ctx*, int64_t, int64_t, int64_t, const int32_t*, const int32_t*, const double*, const double*, bool defer_values);
fmwr_data* data_create_csr32(fmwr_ctx*, int64_t, int64_t, int64_t, const uint32_t*, const uint32_t*, const float*, const float*);

static void fetch_pred(fmwr_ctx* ctx, fmwr_data* d, double* out)
{
  if (d->n == 0) return;
  ctx->d2h_bytes += 8 * d->n;
  if (d->pred_prec == FMWR_F64) {
    FMWR_REQUIRE(d->pred64.p, FMWR_ERR_ARG, "no forward result on the device");
    FMWR_CUDA(cudaMemcpyAsync(out, d->pred64.p, 8 * d->n, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } else {
    FMWR_REQUIRE(d->pred32.p, FMWR_ERR_ARG, "no forward result on the device");
    // widen on the device, fetch doubles (the R side wants a NumericVector)
    DBuf<double> wide;
    wide.alloc(d->n);
    FMWR_LAUNCH(ctx, cast_to_f64<float>, ceil_div(d->n, 256), 256, 0, d->pred32.p, wide.p, d->n);
    FMWR_CUDA(cudaMemcpyAsync(out, wide.p, 8 * d->n, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  }
}

// eval sets of fmwr_train_posterior_dev / fmwr_train_holdout_dev: non-null, labelled if scored, not d, listed once, p features
static void check_eval_list(const fmwr_model* m, const fmwr_data* d, fmwr_data* const* eval, int n_eval, bool need_labels)
{
  for (int i = 0; i < n_eval; ++i) {
    FMWR_REQUIRE(eval[i], FMWR_ERR_ARG, "null eval data");
    FMWR_REQUIRE(!need_labels || eval[i]->has_labels, FMWR_ERR_ARG, "an eval set has no labels");
    FMWR_REQUIRE(eval[i] != d, FMWR_ERR_ARG, "an eval set is the training data");
    for (int j = 0; j < i; ++j) FMWR_REQUIRE(eval[j] != eval[i], FMWR_ERR_ARG, "an eval set appears twice");
  }
  for (int i = 0; i < n_eval; ++i) require_same_features(m, eval[i]);
}

// attribute groups of fmwr_solver_cfg (MCMC, and SGD through fmwr_train_sgda_dev; NULL map: one group)
static void check_groups(const fmwr_model* m, const fmwr_solver_cfg* s, bool grouped_solver)
{
  if (!s->attr_group) {
    FMWR_REQUIRE(s->n_groups >= 0 && s->n_groups <= 1, FMWR_ERR_ARG, "n_groups > 1 needs an attr_group map");
    return;
  }
  FMWR_REQUIRE(grouped_solver, FMWR_ERR_ARG, "attribute groups need the MCMC solver");
  FMWR_REQUIRE(s->n_groups >= 1 && s->n_groups <= 65536 && s->n_groups <= m->p, FMWR_ERR_ARG,
               "n_groups must be at least 1 and at most 65536 and the number of features");
  for (int64_t i = 0; i < m->p; ++i)
    FMWR_REQUIRE(s->attr_group[i] >= 0 && s->attr_group[i] < s->n_groups, FMWR_ERR_ARG, "attr_group entry out of range [0, n_groups)");
}

static void train_dispatch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr,
                           const Posterior* post = nullptr, const Holdout* holdout = nullptr)
{
  FMWR_REQUIRE(d->has_labels, FMWR_ERR_ARG, "target's length is not equal the number of cases...");
  FMWR_REQUIRE(d->p == m->p, FMWR_ERR_SHAPE, "there's no the same number of features between train and fm object...");
  check_groups(m, s, s->solver == FMWR_MCMC);
  if (tr) { tr->n_rec = 0; tr->convergent = 0; tr->iters_done = 0; }
  switch (s->solver) {
    case FMWR_SGD: case FMWR_FTRL: case FMWR_TDAP:
      if (s->mode == FMWR_MODE_MINIBATCH) train_minibatch(ctx, m, d, s, tr, holdout);
      else train_exact(ctx, m, d, s, tr, holdout);
      break;
    case FMWR_ALS: case FMWR_MCMC:
      train_als_mcmc(ctx, m, d, s, tr, post, holdout);
      break;
    default: throw Error(FMWR_ERR_ARG, "Unknown solver...");   // reference src/FM.cpp:85
  }
}

}  // namespace fmwr

using namespace fmwr;

extern "C" {

const char* fmwr_last_error(void) { return g_last_error.c_str(); }
int fmwr_version(void) { return 100; }

int fmwr_ctx_create(int device, fmwr_ctx** out)
{
  return guarded([&] {
    FMWR_REQUIRE(out, FMWR_ERR_ARG, "null out pointer");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) throw Error(FMWR_ERR_CUDA, "no CUDA device: fmwr_b200 has no CPU fallback");
    FMWR_REQUIRE(device >= 0 && device < count, FMWR_ERR_ARG, "device ordinal out of range");
    FMWR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    FMWR_CUDA(cudaGetDeviceProperties(&prop, device));
    FMWR_REQUIRE(prop.major >= 10, FMWR_ERR_UNSUPPORTED, "fmwr_b200 is built for sm_100a (Blackwell) only");
    fmwr_ctx* c = new fmwr_ctx();
    try {
      c->device = device;
      c->sm_count = prop.multiProcessorCount;
      if (prop.sharedMemPerBlockOptin > 0) c->smem_optin = (int)prop.sharedMemPerBlockOptin;
      {
        // the staging stream carries upload chunks and their tiny f64 -> f32 narrowing kernels, one after the other; if such a
        // kernel waits for SM slots behind the compute stream's large grids the whole upload pauses (measured: the key sort
        // delayed the value upload by its own 25 ms).  High priority lets its CTAs in as soon as any CTA retires.
        int prio_lo = 0, prio_hi = 0;
        FMWR_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        FMWR_CUDA(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_lo));
        FMWR_CUDA(cudaStreamCreateWithPriority(&c->copy_stream, cudaStreamNonBlocking, prio_hi));
      }
      FMWR_CUDA(cudaEventCreate(&c->ev0));
      FMWR_CUDA(cudaEventCreate(&c->ev1));
      for (int i = 0; i < 2; ++i) {
        FMWR_CUDA(cudaEventCreateWithFlags(&c->ev_copy[i], cudaEventDisableTiming));
        FMWR_CUDA(cudaEventCreateWithFlags(&c->ev_comp[i], cudaEventDisableTiming));
      }
      build_link_tables(c);
      c->red_scratch.alloc(4096);
      c->h_scalar.ensure(64);
      FMWR_CUDA(cudaStreamSynchronize(c->stream));
    } catch (...) { delete c; throw; }
    *out = c;
  });
}

int fmwr_ctx_destroy(fmwr_ctx* ctx)
{
  return guarded([&] {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (int i = 0; i < 2; ++i) { if (ctx->ev_copy[i]) cudaEventDestroy(ctx->ev_copy[i]); if (ctx->ev_comp[i]) cudaEventDestroy(ctx->ev_comp[i]); }
    for (auto& r : ctx->prof_recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    for (auto& e : ctx->prof_pool) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
  });
}

int fmwr_ctx_sync(fmwr_ctx* ctx)
{
  return guarded([&] { FMWR_REQUIRE(ctx, FMWR_ERR_ARG, "null ctx"); FMWR_CUDA(cudaStreamSynchronize(ctx->stream)); });
}

int fmwr_timer_start(fmwr_ctx* ctx)
{
  return guarded([&] { FMWR_REQUIRE(ctx, FMWR_ERR_ARG, "null ctx"); FMWR_CUDA(cudaEventRecord(ctx->ev0, ctx->stream)); });
}

int fmwr_timer_stop_ms(fmwr_ctx* ctx, double* ms)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && ms, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    FMWR_CUDA(cudaEventSynchronize(ctx->ev1));
    float f = 0;
    FMWR_CUDA(cudaEventElapsedTime(&f, ctx->ev0, ctx->ev1));
    *ms = f;
  });
}

int fmwr_ctx_transfer_bytes(fmwr_ctx* ctx, int64_t* h2d, int64_t* d2h)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx, FMWR_ERR_ARG, "null ctx");
    if (h2d) *h2d = ctx->h2d_bytes;
    if (d2h) *d2h = ctx->d2h_bytes;
  });
}

int fmwr_ctx_launch_count(fmwr_ctx* ctx, int64_t* n)
{
  return guarded([&] { FMWR_REQUIRE(ctx && n, FMWR_ERR_ARG, "null argument"); *n = ctx->launches; });
}

int fmwr_profile_enable(fmwr_ctx* ctx, int on)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx, FMWR_ERR_ARG, "null ctx");
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    for (auto& r : ctx->prof_recs) { ctx->prof_pool.push_back(r.e0); ctx->prof_pool.push_back(r.e1); }
    ctx->prof_recs.clear();
    ctx->profile = on != 0;
  });
}

int fmwr_profile_read(fmwr_ctx* ctx, char* buf, int64_t buf_len)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && buf && buf_len > 0, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    struct Agg { const char* tag; double ms; int64_t n; };
    std::vector<Agg> agg;
    for (auto& r : ctx->prof_recs) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) continue;
      size_t i = 0;
      for (; i < agg.size(); ++i) if (agg[i].tag == r.tag || strcmp(agg[i].tag, r.tag) == 0) break;
      if (i == agg.size()) agg.push_back({r.tag, 0.0, 0});
      agg[i].ms += ms; agg[i].n += 1;
    }
    std::string out;
    for (auto& a : agg) {
      char line[512];
      snprintf(line, sizeof line, "%s\t%lld\t%.6f\n", a.tag, (long long)a.n, a.ms);
      out += line;
    }
    FMWR_REQUIRE((int64_t)out.size() + 1 <= buf_len, FMWR_ERR_ARG, "profile buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
  });
}

int fmwr_mem_trim(void)
{
  return guarded([&] { dev_trim(); });
}

int fmwr_host_pin(void* ptr, int64_t bytes)
{
  return guarded([&] { FMWR_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault)); });
}

int fmwr_host_unpin(void* ptr)
{
  return guarded([&] { FMWR_CUDA(cudaHostUnregister(ptr)); });
}

int fmwr_flush_l2(fmwr_ctx* ctx)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx, FMWR_ERR_ARG, "null ctx");
    const size_t bytes = 256ull << 20;
    ctx->flush_buf.ensure(bytes);
    FMWR_CUDA(cudaMemsetAsync(ctx->flush_buf.p, 1, bytes, ctx->stream));
  });
}

// ---- data ----------------------------------------------------------------------------------------
int fmwr_data_create(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz, const int32_t* row_size, const int32_t* col_idx,
                     const double* value, const double* labels, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && out, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE((n == 0 || row_size) && (nnz == 0 || (col_idx && value)), FMWR_ERR_ARG, "null input array");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    *out = data_create_f64(ctx, n, p, nnz, row_size, col_idx, value, labels, false);
  });
}

int fmwr_data_create_csr32(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz, const uint32_t* rowptr, const uint32_t* col_idx,
                           const float* value, const float* labels, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && out && rowptr, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(nnz == 0 || (col_idx && value), FMWR_ERR_ARG, "null input array");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    *out = data_create_csr32(ctx, n, p, nnz, rowptr, col_idx, value, labels);
  });
}

int fmwr_data_destroy(fmwr_data* d)
{
  return guarded([&] { if (d) { cudaSetDevice(d->ctx->device); delete d; } });
}

int fmwr_data_shape(fmwr_data* d, int64_t* n, int64_t* p, int64_t* nnz)
{
  return guarded([&] {
    FMWR_REQUIRE(d, FMWR_ERR_ARG, "null data");
    if (n) *n = d->n;
    if (p) *p = d->p;
    if (nnz) *nnz = d->nnz;
  });
}

int fmwr_data_get_csr(fmwr_data* d, uint32_t* rowptr, uint32_t* col_idx, float* value, float* labels)
{
  return guarded([&] {
    FMWR_REQUIRE(d, FMWR_ERR_ARG, "null data");
    cudaStream_t s = d->ctx->stream;
    if (rowptr) FMWR_CUDA(cudaMemcpyAsync(rowptr, d->rowptr.p, 4 * (d->n + 1), cudaMemcpyDeviceToHost, s));
    if (col_idx && d->nnz) FMWR_CUDA(cudaMemcpyAsync(col_idx, d->col.p, 4 * d->nnz, cudaMemcpyDeviceToHost, s));
    if (value && d->nnz) FMWR_CUDA(cudaMemcpyAsync(value, d->val.p, 4 * d->nnz, cudaMemcpyDeviceToHost, s));
    if (labels && d->has_labels && d->n) FMWR_CUDA(cudaMemcpyAsync(labels, d->y.p, 4 * d->n, cudaMemcpyDeviceToHost, s));
    FMWR_CUDA(cudaStreamSynchronize(s));
  });
}

int fmwr_data_transpose(fmwr_data* d)
{
  return guarded([&] { FMWR_REQUIRE(d, FMWR_ERR_ARG, "null data"); FMWR_CUDA(cudaSetDevice(d->ctx->device)); transpose_build(d); });
}

int fmwr_data_get_csc(fmwr_data* d, uint32_t* colptr, uint32_t* row_idx, float* value)
{
  return guarded([&] {
    FMWR_REQUIRE(d && d->has_csc, FMWR_ERR_ARG, "no CSC twin: call fmwr_data_transpose first");
    cudaStream_t s = d->ctx->stream;
    if (colptr) FMWR_CUDA(cudaMemcpyAsync(colptr, d->colptr.p, 4 * (d->p + 1), cudaMemcpyDeviceToHost, s));
    if (row_idx && d->nnz) FMWR_CUDA(cudaMemcpyAsync(row_idx, d->crow.p, 4 * d->nnz, cudaMemcpyDeviceToHost, s));
    if (value && d->nnz) FMWR_CUDA(cudaMemcpyAsync(value, d->cval.p, 4 * d->nnz, cudaMemcpyDeviceToHost, s));
    FMWR_CUDA(cudaStreamSynchronize(s));
  });
}

int fmwr_data_scales(fmwr_data* d, const int32_t* norm_cols, int64_t n_norm, double* mean, double* sd)
{
  return guarded([&] {
    FMWR_REQUIRE(d && mean && sd && (n_norm == 0 || norm_cols), FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    data_scales(d, norm_cols, n_norm, mean, sd);
  });
}

int fmwr_data_normalize(fmwr_data* d, const double* mean, const double* sd)
{
  return guarded([&] {
    FMWR_REQUIRE(d && mean && sd, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    data_normalize(d, mean, sd);
  });
}

int fmwr_data_synth(fmwr_ctx* ctx, int64_t n, int32_t n_fields, const int64_t* field_size, const int32_t* skew,
                    int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && out && field_size, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    data_synth(ctx, n, 0, n_fields, field_size, skew, value_mode, label_mode, noise, seed, out);
  });
}

int fmwr_data_synth_rows(fmwr_ctx* ctx, int64_t row_begin, int64_t n_rows, int32_t n_fields, const int64_t* field_size,
                         const int32_t* skew, int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && out && field_size && row_begin >= 0, FMWR_ERR_ARG, "bad argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    data_synth(ctx, n_rows, row_begin, n_fields, field_size, skew, value_mode, label_mode, noise, seed, out);
  });
}

int fmwr_data_slice_columns(fmwr_data* d, int64_t col_begin, int64_t col_end, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(d && out, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    *out = data_slice_columns(d, col_begin, col_end);
  });
}

int fmwr_data_set_labels(fmwr_data* d, const double* labels)
{
  return guarded([&] {
    FMWR_REQUIRE(d && (labels || d->n == 0), FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    data_set_labels(d, labels);
  });
}

int fmwr_data_restore_values(fmwr_data* d)
{
  return guarded([&] {
    FMWR_REQUIRE(d, FMWR_ERR_ARG, "null data");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    data_restore_values(d);
  });
}

int fmwr_data_concat_rows(fmwr_data* const* parts, int32_t n_parts, fmwr_data** out)
{
  return guarded([&] {
    FMWR_REQUIRE(parts && out && n_parts > 0 && parts[0], FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(parts[0]->ctx->device));
    *out = data_concat_rows(parts, n_parts);
  });
}

// ---- model ---------------------------------------------------------------------------------------
int fmwr_model_create(fmwr_ctx* ctx, const fmwr_model_cfg* cfg, int64_t p, int32_t precision, fmwr_model** out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && cfg && out, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(p >= 0 && cfg->k >= 0, FMWR_ERR_ARG, "negative dimension");
    FMWR_REQUIRE(precision == FMWR_F32 || precision == FMWR_F64, FMWR_ERR_ARG, "unknown precision");
    FMWR_REQUIRE(cfg->task == FMWR_CLASSIFICATION || cfg->task == FMWR_REGRESSION, FMWR_ERR_ARG, "unknown task...");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    fmwr_model* m = new fmwr_model();
    try {
      m->ctx = ctx; m->cfg = *cfg; m->p = p; m->prec = precision; m->k = cfg->k;
      m->kp = padded_k(cfg->k, precision);
      m->scal.alloc(64 * sizeof(double));
      m->w.alloc((size_t)(p + 4) * m->esz());            // +4 elements: 16-byte-rounded staging reads (update_tma.cuh)
      m->v.alloc((size_t)p * m->kp * m->esz());
      FMWR_CUDA(cudaMemsetAsync(m->scal.p, 0, m->scal.bytes(), ctx->stream));
      FMWR_CUDA(cudaMemsetAsync(m->w.p, 0, m->w.bytes(), ctx->stream));
      FMWR_CUDA(cudaMemsetAsync(m->v.p, 0, m->v.bytes(), ctx->stream));
      FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    } catch (...) { delete m; throw; }
    *out = m;
  });
}

int fmwr_model_destroy(fmwr_model* m)
{
  return guarded([&] { if (m) { cudaSetDevice(m->ctx->device); delete m; } });
}

int fmwr_model_set(fmwr_model* m, double w0, const double* w, const double* v)
{
  return guarded([&] {
    FMWR_REQUIRE(m && (m->p == 0 || w) && (m->p == 0 || m->k == 0 || v), FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(m->ctx->device));
    model_set_host(m, w0, w, v);
  });
}

int fmwr_model_get(fmwr_model* m, double* w0, double* w, double* v)
{
  return guarded([&] {
    FMWR_REQUIRE(m, FMWR_ERR_ARG, "null model");
    FMWR_CUDA(cudaSetDevice(m->ctx->device));
    model_get_host(m, w0, w, v);
  });
}

int fmwr_model_state_info(fmwr_model* m, int32_t* solver, int32_t* n_state)
{
  return guarded([&] {
    FMWR_REQUIRE(m, FMWR_ERR_ARG, "null model");
    if (solver) *solver = m->state_solver;
    if (n_state) *n_state = m->state_solver ? m->n_state : 0;
  });
}

int fmwr_model_get_state(fmwr_model* m, double* scal8, double* sw, double* sv)
{
  return guarded([&] {
    FMWR_REQUIRE(m, FMWR_ERR_ARG, "null model");
    fmwr_ctx* ctx = m->ctx;
    FMWR_CUDA(cudaSetDevice(ctx->device));
    const int64_t p = m->p;
    if (scal8) FMWR_CUDA(cudaMemcpyAsync(scal8, m->scal.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    const int ns = m->state_solver ? m->n_state : 0;
    DBuf<double> stage;
    stage.alloc(std::max<int64_t>(1, p * (int64_t)std::max(m->k, 1)));
    for (int i = 0; i < ns && p > 0; ++i) {
      if (sw) {
        if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, cast_to_f64<double>, ceil_div(p, 256), 256, 0, (const double*)m->sw[i].p, stage.p, p);
        else FMWR_LAUNCH(ctx, cast_to_f64<float>, ceil_div(p, 256), 256, 0, (const float*)m->sw[i].p, stage.p, p);
        FMWR_CUDA(cudaMemcpyAsync(sw + (size_t)i * p, stage.p, 8 * p, cudaMemcpyDeviceToHost, ctx->stream));
      }
      if (sv && m->k > 0) {
        if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, unpack_v<double>, ceil_div(p * m->k, 256), 256, 0, (const double*)m->sv[i].p, stage.p, p, m->k, m->kp);
        else FMWR_LAUNCH(ctx, unpack_v<float>, ceil_div(p * m->k, 256), 256, 0, (const float*)m->sv[i].p, stage.p, p, m->k, m->kp);
        FMWR_CUDA(cudaMemcpyAsync(sv + (size_t)i * p * m->k, stage.p, 8 * p * m->k, cudaMemcpyDeviceToHost, ctx->stream));
      }
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

int fmwr_model_set_state(fmwr_model* m, int32_t solver, int32_t n_state, const double* scal8, const double* sw, const double* sv)
{
  return guarded([&] {
    FMWR_REQUIRE(m && n_state >= 0 && n_state <= 5, FMWR_ERR_ARG, "bad argument");
    FMWR_REQUIRE(n_state == 0 || (sw && (sv || m->k == 0)), FMWR_ERR_ARG, "null state arrays");
    fmwr_ctx* ctx = m->ctx;
    FMWR_CUDA(cudaSetDevice(ctx->device));
    const int64_t p = m->p;
    model_alloc_state(m, n_state, solver, false);
    if (scal8) FMWR_CUDA(cudaMemcpyAsync((double*)m->scal.p + 1, scal8 + 1, 7 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));   // [0] = w0 stays
    DBuf<double> stage;
    stage.alloc(std::max<int64_t>(1, p * (int64_t)std::max(m->k, 1)));
    for (int i = 0; i < n_state && p > 0; ++i) {
      FMWR_CUDA(cudaMemcpyAsync(stage.p, sw + (size_t)i * p, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
      if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, cast_from_f64<double>, ceil_div(p, 256), 256, 0, stage.p, (double*)m->sw[i].p, p);
      else FMWR_LAUNCH(ctx, cast_from_f64<float>, ceil_div(p, 256), 256, 0, stage.p, (float*)m->sw[i].p, p);
      if (m->k > 0) {
        FMWR_CUDA(cudaMemcpyAsync(stage.p, sv + (size_t)i * p * m->k, 8 * p * m->k, cudaMemcpyHostToDevice, ctx->stream));
        if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, pack_v<double>, ceil_div(p * m->kp, 256), 256, 0, stage.p, (double*)m->sv[i].p, p, m->k, m->kp);
        else FMWR_LAUNCH(ctx, pack_v<float>, ceil_div(p * m->kp, 256), 256, 0, stage.p, (float*)m->sv[i].p, p, m->k, m->kp);
      }
      FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

int fmwr_model_init_random(fmwr_model* m, double mean, double sd, uint64_t seed)
{
  return guarded([&] {
    FMWR_REQUIRE(m, FMWR_ERR_ARG, "null model");
    FMWR_CUDA(cudaSetDevice(m->ctx->device));
    model_init_random(m, mean, sd, seed);
  });
}

// ---- forward -------------------------------------------------------------------------------------
int fmwr_predict_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, int32_t link, double lo, double hi)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    forward_launch(ctx, m, d, link, lo, hi);
  });
}

int fmwr_predict_fetch(fmwr_ctx* ctx, fmwr_data* d, double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && d && (out || d->n == 0), FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    fetch_pred(ctx, d, out);
  });
}

int fmwr_contrib_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(!(ctx->nccl_comm && ctx->world > 1), FMWR_ERR_UNSUPPORTED, "contributions run on one GPU (a column slice holds partial S_f)");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    contrib_launch(ctx, m, d);
  });
}

int fmwr_contrib_fetch(fmwr_ctx* ctx, fmwr_data* d, double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && d && (out || d->nnz == 0), FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(d->contrib64.p, FMWR_ERR_ARG, "no contributions on the device (fmwr_contrib_dev has not run on this data)");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    if (d->nnz == 0) return;
    ctx->d2h_bytes += 8 * d->nnz;
    FMWR_CUDA(cudaMemcpyAsync(out, d->contrib64.p, 8 * d->nnz, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

int fmwr_evaluate_dev(fmwr_ctx* ctx, fmwr_data* d, int32_t task, int32_t metric, double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && d && out, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(d->has_labels, FMWR_ERR_ARG, "data has no labels");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    *out = evaluate_dev(ctx, d, task, metric);
  });
}

int fmwr_train_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d && s, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    train_dispatch(ctx, m, d, s, trace);
  });
}

int fmwr_train_posterior_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace,
                             int32_t burn_in, fmwr_data* const* eval, int32_t n_eval)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d && s, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(n_eval >= 0 && (n_eval == 0 || eval), FMWR_ERR_ARG, "null eval list");
    FMWR_REQUIRE(s->solver == FMWR_MCMC, FMWR_ERR_ARG, "posterior averaging needs the MCMC solver");
    FMWR_REQUIRE(burn_in >= 0 && burn_in < s->max_iter, FMWR_ERR_ARG, "burn_in must be at least 0 and less than max_iter");
    check_eval_list(m, d, eval, n_eval, false);
    FMWR_REQUIRE(!(ctx->nccl_comm && ctx->world > 1), FMWR_ERR_UNSUPPORTED, "posterior averaging runs on one GPU (row-sharded data is not supported)");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    const Posterior post{burn_in, eval, n_eval};
    train_dispatch(ctx, m, d, s, trace, &post);
  });
}

int fmwr_train_holdout_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace,
                           fmwr_data* const* eval, int32_t n_eval, double* eval_scores,
                           int32_t select_best, int32_t patience, int32_t* best_rec)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d && s, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(trace, FMWR_ERR_ARG, "held-out tracking needs a trace (its max_rec bounds the stored scores)");
    FMWR_REQUIRE(s->step_size > 0, FMWR_ERR_ARG, "held-out tracking needs step_size > 0 (the held-out sets are scored at the tracker's records)");
    FMWR_REQUIRE(n_eval >= 1 && eval, FMWR_ERR_ARG, "held-out tracking needs at least one eval set");
    FMWR_REQUIRE(eval_scores, FMWR_ERR_ARG, "null eval_scores");
    FMWR_REQUIRE(patience >= 0, FMWR_ERR_ARG, "patience must be at least 0");
    check_eval_list(m, d, eval, n_eval, true);
    FMWR_REQUIRE(!(ctx->nccl_comm && ctx->world > 1), FMWR_ERR_UNSUPPORTED, "held-out tracking runs on one GPU (sharded models are not supported)");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    int32_t best = -1;
    const Holdout ho{eval, n_eval, eval_scores, trace->max_rec, select_best != 0, patience, &best};
    train_dispatch(ctx, m, d, s, trace, nullptr, &ho);
    if (best_rec) *best_rec = best;
  });
}

int fmwr_train_sgda_dev(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* trace,
                        fmwr_data* valid, double* lambda_w, double* lambda_v)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && m && d && s, FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(s->solver == FMWR_SGD, FMWR_ERR_ARG, "SGDA needs the SGD solver");
    FMWR_REQUIRE(s->mode == FMWR_MODE_EXACT, FMWR_ERR_ARG, "SGDA runs in exact mode only");
    FMWR_REQUIRE(!s->warm_state, FMWR_ERR_ARG, "SGDA starts from zero gradients: warm_state must be 0");
    FMWR_REQUIRE(!(m->cfg.l1_w1 > 0 || m->cfg.l1_v > 0), FMWR_ERR_ARG, "SGDA adapts L2 rates only: L1.w1 and L1.v must be 0");
    FMWR_REQUIRE(d->has_labels, FMWR_ERR_ARG, "target's length is not equal the number of cases...");
    FMWR_REQUIRE(valid, FMWR_ERR_ARG, "null validation data");
    FMWR_REQUIRE(valid != d, FMWR_ERR_ARG, "the validation data is the training data");
    FMWR_REQUIRE(valid->has_labels, FMWR_ERR_ARG, "the validation data has no labels");
    FMWR_REQUIRE(valid->n > 0, FMWR_ERR_ARG, "the validation data has no rows");
    FMWR_REQUIRE(lambda_w && (lambda_v || m->k == 0), FMWR_ERR_ARG, "null lambda_w / lambda_v");
    check_groups(m, s, true);
    const int G = s->attr_group ? s->n_groups : 1;
    for (int g = 0; g < G; ++g) FMWR_REQUIRE(std::isfinite(lambda_w[g]) && lambda_w[g] >= 0, FMWR_ERR_ARG, "lambda_w entries must be finite and >= 0");
    for (int64_t i = 0; i < (int64_t)G * m->k; ++i)
      FMWR_REQUIRE(std::isfinite(lambda_v[i]) && lambda_v[i] >= 0, FMWR_ERR_ARG, "lambda_v entries must be finite and >= 0");
    FMWR_REQUIRE(d->p == m->p, FMWR_ERR_SHAPE, "there's no the same number of features between train and fm object...");
    require_same_features(m, valid);
    FMWR_REQUIRE(!(ctx->nccl_comm && ctx->world > 1), FMWR_ERR_UNSUPPORTED, "SGDA runs on one GPU (sharded models are not supported)");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    if (trace) { trace->n_rec = 0; trace->convergent = 0; trace->iters_done = 0; }
    train_sgda(ctx, m, d, s, trace, valid, lambda_w, lambda_v);
  });
}

// ---- one-shot host entry points ----------------------------------------------------------------
static fmwr_ctx* default_ctx()
{
  static std::mutex mu;
  static fmwr_ctx* ctx = nullptr;
  std::lock_guard<std::mutex> lk(mu);
  if (!ctx) {
    int dev = 0;
    if (const char* e = getenv("FMWR_DEVICE")) dev = atoi(e);
    if (fmwr_ctx_create(dev, &ctx) != 0) throw Error(FMWR_ERR_CUDA, g_last_error);
  }
  return ctx;
}

// FMWR_TRACE=1: wall-clock of the phases of the one-shot entry points (stderr)
// FMWR_TRACE=2: host-side laps only (no device synchronisation: the pipelined one-shot path stays pipelined)
struct PhaseTimer {
  bool on, host_only; std::chrono::steady_clock::time_point t;
  PhaseTimer() : on(getenv("FMWR_TRACE") != nullptr && atoi(getenv("FMWR_TRACE")) == 1),
                 host_only(getenv("FMWR_TRACE") != nullptr && atoi(getenv("FMWR_TRACE")) == 2), t(std::chrono::steady_clock::now()) {}
  void lap(const char* what)
  {
    if (host_only) {
      auto n = std::chrono::steady_clock::now();
      fprintf(stderr, "[fmwr host ] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
      t = n;
      return;
    }
    if (!on) return;
    cudaDeviceSynchronize();
    auto n = std::chrono::steady_clock::now();
    fprintf(stderr, "[fmwr trace] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
    t = n;
  }
};

struct DataGuard { fmwr_data* d = nullptr; ~DataGuard() { if (d) fmwr_data_destroy(d); } };
struct ModelGuard { fmwr_model* m = nullptr; ~ModelGuard() { if (m) fmwr_model_destroy(m); } };

int fmwr_predict(const fmwr_model_cfg* cfg, int32_t precision, int64_t n, int64_t p, int64_t nnz, const int32_t* row_size,
                 const int32_t* col_idx, const double* value, double w0, const double* w, const double* v, int32_t link,
                 double lo, double hi, double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(cfg && (out || n == 0), FMWR_ERR_ARG, "null argument");
    fmwr_ctx* ctx = default_ctx();
    DataGuard dg; ModelGuard mg;
    if (fmwr_data_create(ctx, n, p, nnz, row_size, col_idx, value, nullptr, &dg.d)) throw Error(FMWR_ERR_ARG, g_last_error);
    if (fmwr_model_create(ctx, cfg, p, precision, &mg.m)) throw Error(FMWR_ERR_ARG, g_last_error);
    model_set_host(mg.m, w0, w, v);
    forward_launch(ctx, mg.m, dg.d, link, lo, hi);
    fetch_pred(ctx, dg.d, out);
  });
}

int fmwr_train(const fmwr_model_cfg* cfg, const fmwr_solver_cfg* s, int64_t n, int64_t p, int64_t nnz, const int32_t* row_size,
               const int32_t* col_idx, const double* value, const double* labels, double* w0, double* w, double* v,
               fmwr_trace* trace)
{
  return guarded([&] {
    FMWR_REQUIRE(cfg && s && w0 && labels, FMWR_ERR_ARG, "null argument");
    fmwr_ctx* ctx = default_ctx();
    DataGuard dg; ModelGuard mg;
    PhaseTimer pt;
    FMWR_REQUIRE(value || nnz == 0, FMWR_ERR_ARG, "null argument");
    // minibatch path: the f64 values (60 % of the bytes) keep uploading on the copy stream while the compute stream
    // builds the per-batch CSC keys; each batch waits for its own chunks
    const bool stream = minibatch_streams_values(s);
    // the model goes up first: once the value chunks are queued on the copy engine nothing else gets through until they are done
    if (fmwr_model_create(ctx, cfg, p, s->precision, &mg.m)) throw Error(FMWR_ERR_ARG, g_last_error);
    model_set_host(mg.m, *w0, w, v);
    pt.lap("model create + set");
    dg.d = data_create_f64(ctx, n, p, nnz, row_size, col_idx, value, labels, stream && !pt.on);
    pt.lap("data_create (H2D + narrow)");
    if (stream) {
      minibatch_build(dg.d, (s->compat & FMWR_COMPAT_SKIP_ROW0) ? 1 : 0, s->batch_size);
      pt.lap("per-batch CSC build");
    }
    train_dispatch(ctx, mg.m, dg.d, s, trace);
    pt.lap("train");
    model_get_host(mg.m, w0, w, v);
    pt.lap("model get (D2H)");
  });
}

int fmwr_transpose(int64_t n, int64_t p, int64_t nnz, const int32_t* row_size, const int32_t* col_idx, const double* value,
                   uint32_t* colptr, uint32_t* row_idx, float* out_value)
{
  return guarded([&] {
    fmwr_ctx* ctx = default_ctx();
    DataGuard dg;
    if (fmwr_data_create(ctx, n, p, nnz, row_size, col_idx, value, nullptr, &dg.d)) throw Error(FMWR_ERR_ARG, g_last_error);
    transpose_build(dg.d);
    if (fmwr_data_get_csc(dg.d, colptr, row_idx, out_value)) throw Error(FMWR_ERR_ARG, g_last_error);
  });
}

int fmwr_track(const fmwr_model_cfg* cfg, int32_t solver, int32_t precision, int64_t n, int64_t p, int64_t nnz,
               const int32_t* row_size, const int32_t* col_idx, const double* value, const double* labels, int32_t n_snap,
               const double* snap_w0, const double* snap_w, const double* snap_v, int32_t metric, double lo, double hi,
               double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(cfg && labels && (n_snap == 0 || (snap_w0 && out)), FMWR_ERR_ARG, "null argument");
    fmwr_ctx* ctx = default_ctx();
    DataGuard dg; ModelGuard mg;
    if (fmwr_data_create(ctx, n, p, nnz, row_size, col_idx, value, labels, &dg.d)) throw Error(FMWR_ERR_ARG, g_last_error);
    if (fmwr_model_create(ctx, cfg, p, precision, &mg.m)) throw Error(FMWR_ERR_ARG, g_last_error);
    // Tracker::report (reference src/core/Tracker.h:70-94): forward + metric per snapshot
    const int link = tracker_link(cfg->task, solver);
    std::vector<double> zw(p > 0 ? p : 1, 0.0), zv((size_t)(p > 0 ? p : 1) * (cfg->k > 0 ? cfg->k : 1), 0.0);
    for (int i = 0; i < n_snap; ++i) {
      const double* wi = snap_w ? snap_w + (size_t)i * p : zw.data();
      const double* vi = snap_v ? snap_v + (size_t)i * p * cfg->k : zv.data();
      model_set_host(mg.m, snap_w0[i], wi, vi);
      forward_launch(ctx, mg.m, dg.d, link, lo, hi);
      out[i] = evaluate_dev(ctx, dg.d, cfg->task, metric);
    }
  });
}

int fmwr_link_table_eval(fmwr_ctx* ctx, int32_t which, int64_t n, const double* x, double* out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && x && out, FMWR_ERR_ARG, "null argument");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    link_table_eval(ctx, which, n, x, out);
  });
}

int fmwr_sort_pairs(fmwr_ctx* ctx, int32_t key_bytes, int64_t n, int32_t bits, const void* keys_in, void* keys_out, uint32_t* perm_out)
{
  return guarded([&] {
    FMWR_REQUIRE(ctx && (n == 0 || (keys_in && keys_out && perm_out)), FMWR_ERR_ARG, "null argument");
    FMWR_REQUIRE(key_bytes == 4 || key_bytes == 8, FMWR_ERR_ARG, "key_bytes must be 4 or 8");
    FMWR_REQUIRE(n >= 0 && bits >= 1 && bits <= 8 * key_bytes, FMWR_ERR_ARG, "bad size / bit count");
    FMWR_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return;
    DBuf<char> kin, kout;
    DBuf<uint32_t> perm;
    kin.alloc((size_t)n * key_bytes); kout.alloc((size_t)n * key_bytes); perm.alloc(n);
    FMWR_CUDA(cudaMemcpyAsync(kin.p, keys_in, (size_t)n * key_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (key_bytes == 4) sort_pairs_u32(ctx, (const uint32_t*)kin.p, (uint32_t*)kout.p, nullptr, perm.p, n, bits);
    else sort_pairs_u64(ctx, (const uint64_t*)kin.p, (uint64_t*)kout.p, nullptr, perm.p, n, bits);
    FMWR_CUDA(cudaMemcpyAsync(keys_out, kout.p, (size_t)n * key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaMemcpyAsync(perm_out, perm.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

int fmwr_data_minibatch_info(fmwr_data* d, int32_t batch_size, int32_t compat, int64_t* n_batches, int64_t* n_segments, int64_t* n_entries)
{
  return guarded([&] {
    FMWR_REQUIRE(d && batch_size > 0, FMWR_ERR_ARG, "bad argument");
    FMWR_CUDA(cudaSetDevice(d->ctx->device));
    minibatch_build(d, (compat & FMWR_COMPAT_SKIP_ROW0) ? 1 : 0, batch_size);
    const int64_t nb = (int64_t)d->mb_batch_seg.size() - 1;
    if (n_batches) *n_batches = nb;
    if (n_segments) *n_segments = nb >= 0 ? d->mb_batch_seg[nb] : 0;
    if (n_entries) *n_entries = minibatch_entries(d);
  });
}

}  // extern "C"
