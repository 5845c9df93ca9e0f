// Device-resident sparse data: CSR ingest, CSR->CSC twin, coordinate phases, per-batch CSC,
// z-score normalisation and the synthetic generators.
//
// Replaces SMatrix<float>::assign / transpose / scales / normalize (reference
// src/util/Smatrix.h:44-61, :155-185, :98-153) and Data::add_data/add_target (src/core/Data.h:48-86).
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include "common.cuh"

#include <algorithm>
#include <cmath>

namespace fmwr {

// ------------------------------------------------------------------------------------------ scan
// exclusive prefix sum of u32 (reduce-then-scan, 3 phases, recursive on the block sums)
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void scan_tile_sums(const uint32_t* __restrict__ in, int64_t n, uint32_t* __restrict__ sums)
{
  __shared__ uint32_t red[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  uint32_t s = 0;
  for (int i = threadIdx.x; i < SCAN_TILE; i += SCAN_THREADS) {
    const int64_t j = base + i;
    if (j < n) s += in[j];
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int i = 0; i < SCAN_THREADS / 32; ++i) t += red[i];
    sums[blockIdx.x] = t;
  }
}

// out[j] = offset[tile] + exclusive scan within tile; out may alias in
__global__ void scan_tile_apply(const uint32_t* __restrict__ in, int64_t n, const uint32_t* __restrict__ tile_off,
                                uint32_t* __restrict__ out)
{
  __shared__ uint32_t warp_tot[SCAN_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t x[SCAN_ITEMS];
  uint32_t t = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    const int64_t j = base + i;
    x[i] = j < n ? in[j] : 0u;
    t += x[i];
  }
  // inclusive scan of per-thread totals across the block
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t inc = t;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  uint32_t woff = 0;
  for (int i = 0; i < wid; ++i) woff += warp_tot[i];
  uint32_t run = tile_off[blockIdx.x] + woff + inc - t;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    const int64_t j = base + i;
    if (j < n) out[j] = run;
    run += x[i];
  }
}

// exclusive scan of in[0..n) into out[0..n); returns nothing (total = out[n-1] + in[n-1])
static void exclusive_scan_u32(fmwr_ctx* ctx, const uint32_t* in, uint32_t* out, int64_t n)
{
  if (n <= 0) return;
  const int64_t tiles = ceil_div64(n, SCAN_TILE);
  DBuf<uint32_t> sums;
  sums.alloc(tiles);
  FMWR_LAUNCH(ctx, scan_tile_sums, (int)tiles, SCAN_THREADS, 0, in, n, sums.p);
  if (tiles > 1) exclusive_scan_u32(ctx, sums.p, sums.p, tiles);
  else FMWR_CUDA(cudaMemsetAsync(sums.p, 0, sizeof(uint32_t), ctx->stream));
  FMWR_LAUNCH(ctx, scan_tile_apply, (int)tiles, SCAN_THREADS, 0, in, n, sums.p, out);
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));   // sums is freed on return
}

// ------------------------------------------------------------------------------------------ ingest
__global__ void f64_to_f32(const double* __restrict__ in, float* __restrict__ out, int64_t n)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)in[i];
}

// flags[0] |= 1 if any col >= p; flags[0] |= 2 if a row is not strictly ascending
__global__ void validate_csr(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, int64_t n,
                             uint32_t p, uint32_t nnz, int* __restrict__ flags)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t b = rowptr[r], e = rowptr[r + 1];
  if (e < b || e > nnz) { atomicOr(flags, 4); return; }
  int bad = 0;
  uint32_t prev = 0;
  for (uint32_t j = b; j < e; ++j) {
    const uint32_t c = col[j];
    if (c >= p) bad |= 1;
    if (j > b && c <= prev) bad |= 2;
    prev = c;
  }
  if (bad) atomicOr(flags, bad);
}

static void finish_create(fmwr_data* d)
{
  fmwr_ctx* ctx = d->ctx;
  if (d->n == 0) return;
  DBuf<int> flags;
  flags.alloc(1);
  flags.zero(ctx->stream);
  FMWR_LAUNCH(ctx, validate_csr, ceil_div(d->n, 256), 256, 0, d->rowptr.p, d->col.p, d->n, (uint32_t)d->p,
              (uint32_t)d->nnz, flags.p);
  int h = 0;
  FMWR_CUDA(cudaMemcpyAsync(&h, flags.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  FMWR_REQUIRE(!(h & 4), FMWR_ERR_SHAPE, "the length of input's row_size is not correct...");
  FMWR_REQUIRE(!(h & 1), FMWR_ERR_SHAPE, "col_idx out of range (>= number of features)");
  FMWR_REQUIRE(!(h & 2), FMWR_ERR_SHAPE, "col_idx must be strictly ascending within each row");
}

static void set_labels(fmwr_data* d, const float* y)
{
  d->has_labels = true;
  d->y.alloc(d->n);
  FMWR_CUDA(cudaMemcpyAsync(d->y.p, y, sizeof(float) * d->n, cudaMemcpyHostToDevice, d->ctx->stream));
  // Data::add_target min/max (reference src/core/Data.h:80-84)
  float mn = INFINITY, mx = -INFINITY;
  for (int64_t i = 0; i < d->n; ++i) { mn = std::min(mn, y[i]); mx = std::max(mx, y[i]); }
  d->min_y = mn; d->max_y = mx;
  FMWR_CUDA(cudaStreamSynchronize(d->ctx->stream));
}

// labels: f64 -> f32 on the device and Data::add_target's min / max (reference src/core/Data.h:80-84) by a device reduction
__global__ void labels_narrow_minmax(const double* __restrict__ in, float* __restrict__ out, int64_t n, float* __restrict__ mm)
{
  __shared__ float smn[8], smx[8];
  float mn = INFINITY, mx = -INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float y = (float)in[i];
    out[i] = y;
    mn = fminf(mn, y); mx = fmaxf(mx, y);
  }
  for (int o = 16; o > 0; o >>= 1) { mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
  if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) { mn = fminf(mn, smn[i]); mx = fmaxf(mx, smx[i]); }
    mm[2 * blockIdx.x] = mn; mm[2 * blockIdx.x + 1] = mx;
  }
}

static void set_labels_f64(fmwr_data* d, const double* labels)
{
  fmwr_ctx* ctx = d->ctx;
  const int64_t n = d->n;
  d->has_labels = true;
  d->y.alloc(n);
  d->min_y = INFINITY; d->max_y = -INFINITY;
  if (n == 0) return;
  DBuf<double> stage;
  stage.alloc(n);
  const int nblk = (int)std::min<int64_t>(512, ceil_div64(n, 256));
  DBuf<float> mm;
  mm.alloc(2 * (size_t)nblk);
  FMWR_CUDA(cudaMemcpyAsync(stage.p, labels, 8 * n, cudaMemcpyHostToDevice, ctx->stream));
  FMWR_LAUNCH(ctx, labels_narrow_minmax, nblk, 256, 0, stage.p, d->y.p, n, mm.p);
  std::vector<float> h(2 * (size_t)nblk);
  FMWR_CUDA(cudaMemcpyAsync(h.data(), mm.p, 8 * (size_t)nblk, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  float mn = INFINITY, mx = -INFINITY;
  for (int b = 0; b < nblk; ++b) { mn = std::min(mn, h[2 * b]); mx = std::max(mx, h[2 * b + 1]); }
  d->min_y = mn; d->max_y = mx;
}

// entries [lo, hi) of `val` on the compute stream: only the chunks of a mixed upload that came up as raw f64 have anything to
// narrow (the caller has made the stream wait for their events)
static void data_narrow_values(fmwr_data* d, int64_t lo, int64_t hi)
{
  if (!d->val64.p || hi <= lo) return;
  for (int64_t c = lo / d->val_chunk; c * d->val_chunk < hi && c < (int64_t)d->val_dev.size(); ++c) {
    if (!d->val_dev[c]) continue;
    const int64_t a = std::max(lo, c * d->val_chunk), b = std::min(hi, std::min(d->nnz, (c + 1) * d->val_chunk));
    if (b <= a) continue;
    f64_to_f32<<<ceil_div(b - a, 256), 256, 0, d->ctx->stream>>>(d->val64.p + a, d->val.p + a, b - a);
    d->ctx->launches++;
    FMWR_CUDA(cudaGetLastError());
  }
}

// host wait until the uploader has QUEUED chunk ci (its copy and its event): only then may a stream wait on the event
static void data_wait_chunk_issued(fmwr_data* d, int64_t ci)
{
  while (d->up_chunks > 0 && d->up_issued.load(std::memory_order_acquire) <= ci) std::this_thread::yield();
}

// every column chunk in, CSR validated: what any reader of `col` other than the per-batch CSC build calls first
static void data_wait_cols(fmwr_data* d)
{
  if (!d->cols_pending) return;
  for (cudaEvent_t e : d->col_ev) FMWR_CUDA(cudaStreamWaitEvent(d->ctx->stream, e, 0));
  d->cols_pending = false;
  finish_create(d);
}

// every value in `val` for the compute stream: what any reader of `val` other than the per-batch value fill calls first
static void data_wait_values(fmwr_data* d)
{
  if (d->up_thread.joinable()) d->up_thread.join();
  if (d->val_ready) FMWR_CUDA(cudaStreamWaitEvent(d->ctx->stream, d->val_ready, 0));
  if (!d->val_all_narrowed) { data_narrow_values(d, 0, d->nnz); d->val_all_narrowed = true; }
}

// f64 -> f32 on the HOST, several threads, into pinned staging; then the f32 chunk crosses PCIe (half the bytes of the value
// stream: at configs[1] 1.56 GB instead of 3.12 GB of a 5.06 GB upload).  Runs in a background thread so the caller can go on
// queueing work (the per-batch CSC build needs only the column ids); chunk c's event is recorded right after its copy.
static void narrow_slice(const double* in, float* out, int64_t n)
{
  int64_t i = 0;
#if defined(__SSE2__)
  // streaming stores: the staging buffer is written once and read by the DMA engine, so the read-for-ownership of a cached store
  // (4 of the 16 bytes of host memory traffic per value) is pure loss; cvtpd2ps rounds like the cast (MXCSR: nearest even)
  while (i < n && (reinterpret_cast<uintptr_t>(out + i) & 15)) { out[i] = (float)in[i]; ++i; }
  for (; i + 4 <= n; i += 4) {
    const __m128 lo = _mm_cvtpd_ps(_mm_loadu_pd(in + i)), hi = _mm_cvtpd_ps(_mm_loadu_pd(in + i + 2));
    _mm_stream_ps(out + i, _mm_movelh_ps(lo, hi));
  }
  _mm_sfence();
#endif
  for (; i < n; ++i) out[i] = (float)in[i];
}

static void start_value_upload(fmwr_data* d, const double* value, int64_t chunk)
{
  fmwr_ctx* ctx = d->ctx;
  const int64_t nnz = d->nnz;
  const int64_t n_chunks = ceil_div64(nnz, chunk);
  ctx->h_stage[0].ensure((size_t)std::min(chunk, nnz));
  ctx->h_stage[1].ensure((size_t)std::min(chunk, nnz));
  for (int64_t c = 0; c < n_chunks; ++c) {
    cudaEvent_t ce = nullptr;
    FMWR_CUDA(cudaEventCreateWithFlags(&ce, cudaEventDisableTiming));
    d->val_ev.push_back(ce);
  }
  FMWR_CUDA(cudaEventCreateWithFlags(&d->val_ready, cudaEventDisableTiming));
  d->val_chunk = chunk;
  d->up_chunks = n_chunks;
  d->up_issued.store(0, std::memory_order_release);
  static const int n_workers = std::max(1, std::min((int)std::thread::hardware_concurrency(), 32));
  const int dev = ctx->device;
  cudaStream_t vs = ctx->copy_stream;
  float* stage[2] = {ctx->h_stage[0].p, ctx->h_stage[1].p};
  // Mixed upload.  Narrowing on the host halves the PCIe bytes but is bound by the host's memory bandwidth (read 8 B, write 4 B per
  // value: 57 ms for configs[1]'s 390M values on this box -- exactly what the raw f64 stream takes on PCIe).  The two resources
  // are independent, so every third chunk goes up RAW (8 B per value, straight from the caller's pinned buffer, no host work)
  // while the host narrows the two chunks before it: PCIe carries 2 x 4 + 8 bytes per three values in the time the host
  // narrows two -- both ~4.7 ms per three 16M-value chunks.  Raw chunks are narrowed on the device by their first reader
  // (data_narrow_values).  Only when the caller's buffer is pinned: a pageable source would be staged by the driver.
  constexpr int P = 3;                       // one raw chunk per P
  bool mix = false;
  if (n_chunks >= P) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, value) == cudaSuccess && at.type == cudaMemoryTypeHost) mix = true;
    cudaGetLastError();
  }
  d->val_dev.assign(n_chunks, 0);
  if (mix) {
    for (int64_t c = P - 1; c < n_chunks; c += P) d->val_dev[c] = 1;
    d->val64.alloc(nnz);
    d->val_all_narrowed = false;
  }
  d->val_waited = 0;
  d->up_thread = std::thread([d, value, chunk, nnz, n_chunks, dev, vs, stage] {
    cudaSetDevice(dev);
    int64_t last_use[2] = {-1, -1};            // the chunk whose copy last read each staging buffer
    int hcount = 0;
    for (int64_t c0 = 0; c0 < n_chunks; c0 += P) {
      // the raw chunk of the triple goes up in two halves, one behind each narrowed chunk's copy: while the host narrows the next
      // chunk (2.4 ms) the link carries 1.15 ms of f32 and 1.15 ms of raw f64 -- neither side waits for the other
      const int64_t cd = c0 + P - 1;
      const bool has_d = cd < n_chunks && d->val_dev[cd];
      const int64_t d_off = cd * chunk, d_m = has_d ? std::min(chunk, nnz - d_off) : 0;
      const int parts = P - 1;                 // one part behind each narrowed chunk
      int d_sent = 0;
      auto send_raw = [&](bool all) {
        if (!has_d || d_sent >= parts) return;
        const int64_t from = d_m * d_sent / parts;
        const int upto = all ? parts : d_sent + 1;
        const int64_t to = d_m * upto / parts;
        if (to > from) cudaMemcpyAsync(d->val64.p + d_off + from, value + d_off + from, sizeof(double) * (to - from), cudaMemcpyHostToDevice, vs);
        d_sent = upto;
        if (d_sent >= parts) cudaEventRecord(d->val_ev[cd], vs);
      };
      for (int64_t c = c0; c < std::min(n_chunks, c0 + P); ++c) {
        if (d->val_dev[c]) continue;
        const int64_t off = c * chunk, m = std::min(chunk, nnz - off);
        const int sb = hcount++ & 1;
        float* buf = stage[sb];
        if (last_use[sb] >= 0) cudaEventSynchronize(d->val_ev[last_use[sb]]);
        last_use[sb] = c;
        const int T = (int)std::min<int64_t>(n_workers, std::max<int64_t>(1, m / 65536));
        std::vector<std::thread> pool;
        const int64_t per = (m + T - 1) / T;
        for (int t = 1; t < T; ++t) {
          const int64_t lo = t * per, hi = std::min(m, lo + per);
          if (lo < hi) pool.emplace_back(narrow_slice, value + off + lo, buf + lo, hi - lo);
        }
        narrow_slice(value + off, buf, std::min(m, per));
        for (auto& th : pool) th.join();
        cudaMemcpyAsync(d->val.p + off, buf, sizeof(float) * m, cudaMemcpyHostToDevice, vs);
        cudaEventRecord(d->val_ev[c], vs);
        send_raw(false);
      }
      send_raw(true);
      d->up_issued.store(std::min(n_chunks, c0 + P), std::memory_order_release);     // the period's copies and events are queued
    }
    cudaEventRecord(d->val_ready, vs);
    d->up_issued.store(n_chunks + 1, std::memory_order_release);
  });
}

fmwr_data* data_create_f64(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz, const int32_t* row_size,
                           const int32_t* col_idx, const double* value, const double* labels, bool defer_values)
{
  FMWR_REQUIRE(n >= 0 && p >= 0 && nnz >= 0, FMWR_ERR_ARG, "negative dimension");
  FMWR_REQUIRE(nnz < (int64_t)0xffffffffll && n < (int64_t)0xffffffffll && p < (int64_t)0xffffffffll, FMWR_ERR_UNSUPPORTED,
               "dimensions must fit 32-bit indices per device shard");
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = n; d->p = p; d->nnz = nnz;
    d->rowptr.alloc(n + 1);
    d->col.alloc(nnz);
    d->val.alloc(nnz);
    // rowptr: prefix sum of row_size on the device (reference src/util/Smatrix.h:55-60)
    FMWR_CUDA(cudaMemsetAsync(d->rowptr.p, 0, sizeof(uint32_t) * (n + 1), ctx->stream));
    if (n > 0) {
      DBuf<uint32_t> rs;
      rs.alloc(n + 1);
      FMWR_CUDA(cudaMemsetAsync(rs.p, 0, sizeof(uint32_t) * (n + 1), ctx->stream));
      FMWR_CUDA(cudaMemcpyAsync(rs.p, row_size, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
      exclusive_scan_u32(ctx, rs.p, d->rowptr.p, n + 1);
      uint32_t total = 0;
      FMWR_CUDA(cudaMemcpy(&total, d->rowptr.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost));
      FMWR_REQUIRE((int64_t)total == nnz, FMWR_ERR_SHAPE, "the length of input's row_size is not correct...");
    }
    // the labels first: a copy queued behind the column chunks would sit on the copy engine (and the host in its sync) until
    // all of them are through
    if (labels) set_labels_f64(d, labels);
    if (nnz > 0) {
      const int64_t chunk_env = getenv("FMWR_VAL_CHUNK") ? atoll(getenv("FMWR_VAL_CHUNK")) : 0;      // read per call: tests shrink it
      const int64_t chunk = chunk_env > 0 ? chunk_env : (16ll << 20);
      if (defer_values) {
        // one-shot training: the column ids go up in chunks on the copy stream, one event each, and nobody waits here -- the
        // per-batch CSC of a row group is built as soon as its chunks are in (minibatch_build)
        for (int64_t off = 0; off < nnz; off += chunk) {
          const int64_t mm = std::min(chunk, nnz - off);
          FMWR_CUDA(cudaMemcpyAsync(d->col.p + off, col_idx + off, sizeof(int32_t) * mm, cudaMemcpyHostToDevice, ctx->copy_stream));
          cudaEvent_t ce = nullptr;
          FMWR_CUDA(cudaEventCreateWithFlags(&ce, cudaEventDisableTiming));
          FMWR_CUDA(cudaEventRecord(ce, ctx->copy_stream));
          d->col_ev.push_back(ce);
        }
        d->col_chunk = chunk;
        d->cols_pending = true;
      } else {
        FMWR_CUDA(cudaMemcpyAsync(d->col.p, col_idx, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice, ctx->stream));
      }
      // defer_values: nobody waits for the values here -- the one-shot training path sorts the (batch, feature) keys (which need
      // only rowptr and col) while the values are still crossing PCIe, and each batch waits for its own chunks before it reads them
      FMWR_CUDA(cudaEventRecord(ctx->ev_copy[0], ctx->stream));        // the column ids go first: the key sort needs all of them
      FMWR_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[0], 0));
      start_value_upload(d, value, chunk);
      if (!defer_values) { data_wait_values(d); FMWR_CUDA(cudaStreamSynchronize(ctx->stream)); }
    }
    {
      int64_t vbytes = 4 * nnz;                                            // values cross as f32, narrowed on the host ...
      for (size_t c = 0; c < d->val_dev.size(); ++c)                       // ... except the chunks of a mixed upload that go up raw
        if (d->val_dev[c]) vbytes += 4 * std::min<int64_t>(d->val_chunk, nnz - (int64_t)c * d->val_chunk);
      ctx->h2d_bytes += 4 * n + 4 * nnz + vbytes + (labels ? 8 * n : 0);
    }
    if (!d->cols_pending) finish_create(d);            // (chunked columns: validated by the per-batch CSC build, or by data_wait_cols)
  } catch (...) { delete d; throw; }
  return d;
}

fmwr_data* data_create_csr32(fmwr_ctx* ctx, int64_t n, int64_t p, int64_t nnz, const uint32_t* rowptr,
                             const uint32_t* col_idx, const float* value, const float* labels)
{
  FMWR_REQUIRE(n >= 0 && p >= 0 && nnz >= 0, FMWR_ERR_ARG, "negative dimension");
  FMWR_REQUIRE(nnz < (int64_t)0xffffffffll && n < (int64_t)0xffffffffll && p < (int64_t)0xffffffffll, FMWR_ERR_UNSUPPORTED,
               "dimensions must fit 32-bit indices per device shard");
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = n; d->p = p; d->nnz = nnz;
    d->rowptr.alloc(n + 1); d->col.alloc(nnz); d->val.alloc(nnz);
    FMWR_CUDA(cudaMemcpyAsync(d->rowptr.p, rowptr, sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, ctx->stream));
    if (nnz > 0) {
      FMWR_CUDA(cudaMemcpyAsync(d->col.p, col_idx, sizeof(uint32_t) * nnz, cudaMemcpyHostToDevice, ctx->stream));
      FMWR_CUDA(cudaMemcpyAsync(d->val.p, value, sizeof(float) * nnz, cudaMemcpyHostToDevice, ctx->stream));
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    FMWR_REQUIRE(rowptr[n] == (uint32_t)nnz && rowptr[0] == 0, FMWR_ERR_SHAPE, "the length of input's row_size is not correct...");
    if (labels) set_labels(d, labels);
    ctx->h2d_bytes += 4 * (n + 1) + 8 * nnz + (labels ? 4 * n : 0);
    finish_create(d);
  } catch (...) { delete d; throw; }
  return d;
}

// ------------------------------------------------------------------------------------------ CSR -> CSC
__global__ void expand_rows(const uint32_t* __restrict__ rowptr, int64_t n, uint32_t* __restrict__ erow)
{
  // one warp per row writes the row id over the row's entry range
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const uint32_t b = rowptr[row], e = rowptr[row + 1];
  for (uint32_t j = b + (threadIdx.x & 31); j < e; j += 32) erow[j] = (uint32_t)row;
}

__global__ void iota_u32(uint32_t* __restrict__ a, int64_t n)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = (uint32_t)i;
}

__global__ void gather_csc(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ erow, const float* __restrict__ val,
                           int64_t nnz, uint32_t* __restrict__ crow, float* __restrict__ cval)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t e = perm[i];
  crow[i] = erow[e];
  cval[i] = val[e];
}

// ptr[c] = first index i with keys[i] >= c  (keys sorted ascending), c in [0, p]
__global__ void segment_ptr_from_sorted(const uint32_t* __restrict__ keys, int64_t nnz, int64_t p, uint32_t* __restrict__ ptr)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > nnz) return;
  const int64_t lo = (i == 0) ? 0 : (int64_t)keys[i - 1] + 1;
  const int64_t hi = (i == nnz) ? p : (int64_t)keys[i];
  for (int64_t c = lo; c <= hi; ++c) ptr[c] = (uint32_t)i;
}

static int bits_for(uint64_t maxval)
{
  int b = 1;
  while (b < 64 && (maxval >> b) != 0) ++b;
  return b;
}

// stable sort of entry ids by column: radix sort keeps equal keys in input (== row-ascending) order
void transpose_build(fmwr_data* d)
{
  if (d->has_csc) return;
  fmwr_ctx* ctx = d->ctx;
  const int64_t nnz = d->nnz, n = d->n, p = d->p;
  d->colptr.alloc(p + 1);
  d->crow.alloc(nnz);
  d->cval.alloc(nnz);
  if (nnz == 0) {
    FMWR_CUDA(cudaMemsetAsync(d->colptr.p, 0, sizeof(uint32_t) * (p + 1), ctx->stream));
    d->has_csc = true;
    return;
  }
  DBuf<uint32_t> erow, keys_out, idx_out;
  erow.alloc(nnz); keys_out.alloc(nnz); idx_out.alloc(nnz);
  FMWR_LAUNCH(ctx, expand_rows, ceil_div(n * 32, 256), 256, 0, d->rowptr.p, n, erow.p);
  const int end_bit = bits_for((uint64_t)(p > 0 ? p - 1 : 0));
  sort_pairs_u32(ctx, d->col.p, keys_out.p, nullptr, idx_out.p, nnz, end_bit);      // values = entry ids 0 .. nnz-1 (sort.cu)
  FMWR_LAUNCH(ctx, gather_csc, ceil_div(nnz, 256), 256, 0, idx_out.p, erow.p, d->val.p, nnz, d->crow.p, d->cval.p);
  FMWR_LAUNCH(ctx, segment_ptr_from_sorted, ceil_div(nnz + 1, 256), 256, 0, keys_out.p, nnz, p, d->colptr.p);
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  d->has_csc = true;
}

void launch_iota(fmwr_ctx* ctx, uint32_t* a, int64_t n)
{
  if (n > 0) FMWR_LAUNCH(ctx, iota_u32, ceil_div(n, 256), 256, 0, a, n);
}

// ------------------------------------------------------------------------------------------ phases
// prev[c] = max over rows containing c of the column that precedes c in that row (+1; 0 = none).
__global__ void phase_prev(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, int64_t n,
                           uint32_t* __restrict__ prev)
{
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const uint32_t b = rowptr[row], e = rowptr[row + 1];
  for (uint32_t j = b + 1 + (threadIdx.x & 31); j < e; j += 32) atomicMax(prev + col[j], col[j - 1] + 1u);
}

// Greedy split of the feature axis into consecutive ranges whose members never co-occur in a row.
// Updating all features of such a range concurrently equals the reference's sequential Gauss-Seidel
// sweep (src/solver/MCMC_ALS_Learner.h:211-255, :303-351 at nthreads=1) because their column
// supports -- the only entries of e and q they touch -- are disjoint.
void phases_build(fmwr_data* d)
{
  if (d->has_phases) return;
  fmwr_ctx* ctx = d->ctx;
  const int64_t p = d->p, n = d->n;
  DBuf<uint32_t> prev;
  prev.alloc(p);
  prev.zero(ctx->stream);
  if (n > 0) FMWR_LAUNCH(ctx, phase_prev, ceil_div(n * 32, 256), 256, 0, d->rowptr.p, d->col.p, n, prev.p);
  // row-sharded data (communicator initialised): the phases must come from the UNION of the shards' rows, or the ranks
  // would disagree on the coordinate steps they all-reduce
  if (ctx->nccl_comm && ctx->world > 1 && p > 0) comm_allreduce_max_u32(ctx, prev.p, (size_t)p);
  std::vector<uint32_t> h(p);
  FMWR_CUDA(cudaMemcpyAsync(h.data(), prev.p, sizeof(uint32_t) * p, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  d->phase_begin.clear();
  d->phase_begin.push_back(0);
  uint32_t a = 0;
  for (int64_t c = 0; c < p; ++c) {
    if (h[c] > a) {            // some row holds c together with a feature >= a of the current range
      a = (uint32_t)c;
      d->phase_begin.push_back(a);
    }
  }
  d->phase_begin.push_back((uint32_t)p);
  d->has_phases = true;
}

// ------------------------------------------------------------------------------------------ per-batch CSC
// Entries of rows [row0, n) regrouped by (batch, feature, row): the "sorted-key segmented reduction" layout of the minibatch update
// kernels (one segment = one touched coordinate).  It is built ROW GROUP BY ROW GROUP: a group is a run of whole batches whose
// entries are sorted on (batch inside the group, feature) and emitted into the global arrays at the group's entry / segment
// offsets.  Resident data is one group.  While the column ids are still uploading (one-shot training path) a group holds ~32M
// entries and is built as soon as its column chunks are in -- fewer key bits, one radix pass less than the whole-matrix sort.
template <class K>
__global__ void mbg_keys(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, int64_t r0, int64_t r1, int64_t row0,
                         uint32_t batch, uint32_t b0, int colbits, uint32_t eg0, K* __restrict__ keys, uint32_t* __restrict__ erow)
{
  const int64_t row = r0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (row >= r1) return;
  const uint32_t b = rowptr[row], e = rowptr[row + 1];
  const uint64_t bid = (uint64_t)((row - row0) / batch) - b0;
  for (uint32_t j = b + (threadIdx.x & 31); j < e; j += 32) {
    keys[j - eg0] = (K)((bid << colbits) | (uint64_t)col[j]);
    erow[j - eg0] = (uint32_t)row;
  }
}

// head[i] = 1 where a new (batch, col) segment starts
template <class K>
__global__ void mb_heads(const K* __restrict__ keys, int64_t m, uint32_t* __restrict__ head)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

// val: the group's values go into ent_val and the segment records.  val == nullptr (values still uploading): the permutation goes
// into perm_global instead, for mb_fill_values to write the values batch by batch once they have arrived.
template <class K>
__global__ void mbg_emit(const K* __restrict__ keys, const uint32_t* __restrict__ head, const uint32_t* __restrict__ segid,
                         const uint32_t* __restrict__ perm_local, const uint32_t* __restrict__ erow, const float* __restrict__ val,
                         int64_t mg, int colbits, uint32_t eg0, uint32_t eoff, uint32_t seg_base, uint32_t n_seg_g,
                         uint32_t* __restrict__ seg_ptr, uint4* __restrict__ seg_rec, uint32_t* __restrict__ ent_row,
                         float* __restrict__ ent_val, uint32_t* __restrict__ perm_global)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= mg) return;
  // every load before the first store: a segment head's loads then share the entry's round trip
  const uint32_t e = perm_local[i];
  const bool h = head[i] != 0;
  const uint32_t r = erow[e];
  const float x = val ? val[eg0 + e] : 0.f;
  const uint32_t s = h ? seg_base + segid[i] : 0u;
  const uint32_t c = h ? (uint32_t)((uint64_t)keys[i] & ((1ull << colbits) - 1ull)) : 0u;
  ent_row[eoff + i] = r;
  if (val) ent_val[eoff + i] = x;
  else perm_global[eoff + i] = e + eoff;             // relative to the first entry of the whole structure
  if (h) {
    // segment record: {feature, length (filled by mb_seg_len), first row, first value} -- one 16-byte load gives
    // the update kernel everything it needs for the common single-entry segment
    seg_ptr[s] = eoff + (uint32_t)i;
    seg_rec[s] = make_uint4(c, 0u, r, __float_as_uint(x));
  }
  if (i == mg - 1) seg_ptr[seg_base + n_seg_g] = eoff + (uint32_t)mg;
}

// values of the segments [seg_lo, seg_hi) (one batch) once their upload has arrived: ent_val and the record's first value
__global__ void mb_fill_values(const uint32_t* __restrict__ seg_ptr, uint4* __restrict__ seg_rec, const uint32_t* __restrict__ perm,
                               const float* __restrict__ val, uint32_t e0, uint32_t seg_lo, uint32_t seg_hi, float* __restrict__ ent_val)
{
  const uint32_t s = seg_lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= seg_hi) return;
  const uint32_t i0 = seg_ptr[s], i1 = seg_ptr[s + 1];
  for (uint32_t i = i0; i < i1; ++i) {
    const float x = val[e0 + perm[i]];
    ent_val[i] = x;
    if (i == i0) seg_rec[s].w = __float_as_uint(x);
  }
}

// device -> pinned host memory by a kernel (zero-copy store over PCIe): no copy engine, so it cannot queue behind uploads
__global__ void peek_u32(const uint32_t* __restrict__ src, int64_t n, uint32_t* __restrict__ host_dst)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) host_dst[i] = src[i];
}
__global__ void peek2_u32(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ host_dst)
{
  if (threadIdx.x == 0 && blockIdx.x == 0) { host_dst[0] = *a; host_dst[1] = *b; }
}

// out[b] = rowptr[min(row0 + b * batch, n)]: the first entry of batch b
__global__ void batch_row_ptr(const uint32_t* __restrict__ rowptr, int64_t row0, int64_t batch, int64_t n, int64_t count, uint32_t* __restrict__ out)
{
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= count) return;
  const int64_t r = row0 + b * batch;
  out[b] = rowptr[r < n ? r : n];
}

__global__ void mb_seg_len(const uint32_t* __restrict__ seg_ptr, uint4* __restrict__ seg_rec, uint32_t n_seg)
{
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_seg) seg_rec[s].y = seg_ptr[s + 1] - seg_ptr[s];
}

// host_dst[k] = segment of the first sorted entry of batch b0 + k (a batch's entries are as many in sorted order as in row order
// and come in batch order); past the group's last entry: its end
__global__ void mbg_batch_first_seg(const uint32_t* __restrict__ batch_ent, uint32_t eg0, const uint32_t* __restrict__ segid, uint32_t mg, uint32_t n_seg_g,
                                    uint32_t seg_base, int64_t b0, int64_t count, uint32_t* __restrict__ host_dst)
{
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const uint32_t i = batch_ent[b0 + k] - eg0;
  host_dst[k] = seg_base + (i < mg ? segid[i] : n_seg_g);
}

template <class K>
static void minibatch_build_grouped(fmwr_data* d, int64_t row0, int64_t batch, int64_t gb /* batches per group */, int gbits)
{
  fmwr_ctx* ctx = d->ctx;
  const bool streaming = d->cols_pending;              // column ids (and values) still crossing PCIe
  const int64_t rows = d->n - row0;
  const int64_t n_batches = ceil_div64(rows, batch);
  d->mb_batch_seg.assign(n_batches + 1, 0);
  // small device -> host reads are zero-copy stores of a kernel into pinned memory: a cudaMemcpy of 4 bytes would queue behind
  // the upload chunks on the copy engine (measured: the build then ends when the upload ends)
  ctx->h_u32.ensure(2 * (size_t)n_batches + 64);
  uint32_t* hp = ctx->h_u32.p;
  DBuf<uint32_t> bp;
  bp.alloc(n_batches + 1);
  FMWR_LAUNCH(ctx, batch_row_ptr, ceil_div(n_batches + 1, 256), 256, 0, d->rowptr.p, row0, batch, d->n, n_batches + 1, bp.p);
  FMWR_LAUNCH(ctx, peek_u32, ceil_div(n_batches + 1, 256), 256, 0, bp.p, n_batches + 1, hp + 8);
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  std::vector<uint32_t> ent(hp + 8, hp + 8 + n_batches + 1);       // absolute first entry of every batch
  const uint32_t e0 = ent[0], e1 = ent[n_batches];
  const int64_t m = (int64_t)e1 - e0;
  // entries before each batch (rows of a batch are consecutive, so this is also the batch's offset in the sorted arrays)
  d->mb_batch_ent.resize(n_batches + 1);
  for (int64_t b = 0; b <= n_batches; ++b) d->mb_batch_ent[b] = (int64_t)ent[b] - (int64_t)e0;
  const int colbits = bits_for((uint64_t)(d->p > 0 ? d->p - 1 : 0));
  // segments: at most one per entry and at most one per (batch, feature)
  const int64_t seg_cap = (int64_t)std::min<uint64_t>(m, (uint64_t)n_batches * (uint64_t)d->p);
  d->mb_ent_row.alloc(m + 8); d->mb_ent_val.alloc(m + 8);      // +8: the dense update kernel stages 16-byte-rounded ranges (update_tma.cuh)
  if (streaming) d->mb_perm.alloc(m);
  else data_wait_values(d);
  int64_t mg_max = 0;
  for (int64_t b0 = 0; b0 < n_batches; b0 += gb) mg_max = std::max<int64_t>(mg_max, (int64_t)ent[std::min(n_batches, b0 + gb)] - ent[b0]);
  DBuf<K> keys_in, keys_out;
  DBuf<uint32_t> perm, erow, head, segid;
  DBuf<int> flags;
  keys_in.alloc(mg_max); keys_out.alloc(mg_max); erow.alloc(mg_max); head.alloc(mg_max); segid.alloc(mg_max); perm.alloc(mg_max);
  if (streaming) { flags.alloc(1); flags.zero(ctx->stream); }
  uint32_t seg_base = 0;
  int64_t next_ev = 0;                                 // column chunks already waited for
  for (int64_t b0 = 0; b0 < n_batches; b0 += gb) {
    const int64_t b1 = std::min(n_batches, b0 + gb);
    const int64_t r0 = row0 + b0 * batch, r1 = std::min(d->n, row0 + b1 * batch);
    const uint32_t eg0 = ent[b0], eg1 = ent[b1];
    const int64_t mg = (int64_t)eg1 - eg0;
    if (streaming) {
      // the chunks that hold this group's column ids
      const int64_t need = mg > 0 ? ((int64_t)eg1 - 1) / d->col_chunk + 1 : next_ev;
      for (; next_ev < need && next_ev < (int64_t)d->col_ev.size(); ++next_ev) FMWR_CUDA(cudaStreamWaitEvent(ctx->stream, d->col_ev[next_ev], 0));
    }
    uint32_t n_seg_g = 0;
    if (mg > 0) {
      // (resident data was validated when it was uploaded)
      if (streaming) FMWR_LAUNCH(ctx, validate_csr, ceil_div(r1 - r0, 256), 256, 0, d->rowptr.p + r0, d->col.p, r1 - r0, (uint32_t)d->p, (uint32_t)d->nnz, flags.p);
      FMWR_LAUNCH(ctx, mbg_keys<K>, ceil_div((r1 - r0) * 32, 256), 256, 0, d->rowptr.p, d->col.p, r0, r1, row0, (uint32_t)batch, (uint32_t)b0, colbits, eg0,
                  keys_in.p, erow.p);
      if (sizeof(K) == 4) sort_pairs_u32(ctx, (const uint32_t*)keys_in.p, (uint32_t*)keys_out.p, nullptr, perm.p, mg, colbits + gbits);
      else sort_pairs_u64(ctx, (const uint64_t*)keys_in.p, (uint64_t*)keys_out.p, nullptr, perm.p, mg, colbits + gbits);
      FMWR_LAUNCH(ctx, mb_heads<K>, ceil_div(mg, 256), 256, 0, keys_out.p, mg, head.p);
      exclusive_scan_u32(ctx, head.p, segid.p, mg);
      FMWR_LAUNCH(ctx, peek2_u32, 1, 32, 0, segid.p + (mg - 1), head.p + (mg - 1), hp);
      if (streaming) FMWR_LAUNCH(ctx, peek_u32, 1, 32, 0, reinterpret_cast<const uint32_t*>(flags.p), (int64_t)1, hp + 4);
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    if (streaming && mg > 0) {
      // a bad group stops the build here, with the reference's message, before its keys are taken for segments
      const uint32_t hf = hp[4];
      if (hf) d->cols_pending = false;
      FMWR_REQUIRE(!(hf & 4), FMWR_ERR_SHAPE, "the length of input's row_size is not correct...");
      FMWR_REQUIRE(!(hf & 1), FMWR_ERR_SHAPE, "col_idx out of range (>= number of features)");
      FMWR_REQUIRE(!(hf & 2), FMWR_ERR_SHAPE, "col_idx must be strictly ascending within each row");
    }
    if (mg > 0) n_seg_g = hp[0] + hp[1];
    FMWR_REQUIRE((int64_t)seg_base + n_seg_g <= seg_cap, FMWR_ERR_SHAPE, "segment count exceeds its bound");
    if (b0 == 0) {
      // one group: exactly its segments; several: the bound (the later groups are not counted yet)
      const int64_t cap = gb == n_batches ? n_seg_g : seg_cap;
      d->mb_seg_ptr.alloc((size_t)cap + 1 + 8); d->mb_seg_rec.alloc(cap);
    }
    if (mg > 0) {
      FMWR_LAUNCH(ctx, mbg_emit<K>, ceil_div(mg, 256), 256, 0, keys_out.p, head.p, segid.p, perm.p, erow.p, streaming ? (const float*)nullptr : d->val.p,
                  mg, colbits, eg0, eg0 - e0, seg_base, n_seg_g, d->mb_seg_ptr.p, d->mb_seg_rec.p, d->mb_ent_row.p, d->mb_ent_val.p, d->mb_perm.p);
      FMWR_LAUNCH(ctx, mb_seg_len, ceil_div(n_seg_g, 256), 256, 0, d->mb_seg_ptr.p + seg_base, d->mb_seg_rec.p + seg_base, n_seg_g);
    }
    FMWR_LAUNCH(ctx, mbg_batch_first_seg, ceil_div(b1 - b0, 256), 256, 0, bp.p, eg0, segid.p, (uint32_t)mg, n_seg_g, seg_base, b0, b1 - b0, hp + 16);
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int64_t b = b0; b < b1; ++b) d->mb_batch_seg[b] = hp[16 + (b - b0)];
    seg_base += n_seg_g;
  }
  const uint32_t n_seg = seg_base;
  // empty batches in the middle share the next non-empty one's first segment; trailing ones start at n_seg
  d->mb_batch_seg[n_batches] = n_seg;
  for (int64_t b = n_batches - 1; b >= 0; --b) if (d->mb_batch_seg[b] > d->mb_batch_seg[b + 1]) d->mb_batch_seg[b] = d->mb_batch_seg[b + 1];
  if (m == 0) FMWR_CUDA(cudaMemsetAsync(d->mb_seg_ptr.p, 0, 4, ctx->stream));
  if (streaming) {
    // rows before row0 (the skipped first row) were not part of any group: validate them with the rest of the checks
    for (; next_ev < (int64_t)d->col_ev.size(); ++next_ev) FMWR_CUDA(cudaStreamWaitEvent(ctx->stream, d->col_ev[next_ev], 0));
    if (row0 > 0) FMWR_LAUNCH(ctx, validate_csr, ceil_div(row0, 256), 256, 0, d->rowptr.p, d->col.p, row0, (uint32_t)d->p, (uint32_t)d->nnz, flags.p);
    int h = 0;
    FMWR_CUDA(cudaMemcpyAsync(&h, flags.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    d->cols_pending = false;
    FMWR_REQUIRE(!(h & 4), FMWR_ERR_SHAPE, "the length of input's row_size is not correct...");
    FMWR_REQUIRE(!(h & 1), FMWR_ERR_SHAPE, "col_idx out of range (>= number of features)");
    FMWR_REQUIRE(!(h & 2), FMWR_ERR_SHAPE, "col_idx must be strictly ascending within each row");
  }
  d->mb_batch = batch; d->mb_row0 = row0;
  d->mb_e0 = e0; d->mb_vals_pending = streaming;
}

void minibatch_build(fmwr_data* d, int64_t row0, int64_t batch)
{
  if (d->mb_batch == batch && d->mb_row0 == row0) return;
  const int64_t rows = d->n - row0;
  if (rows <= 0 || batch <= 0) {
    data_wait_cols(d);
    FMWR_REQUIRE(batch > 0, FMWR_ERR_ARG, "batch_size must be positive");
    d->mb_batch_seg.assign(1, 0); d->mb_batch_ent.assign(1, 0);
    d->mb_batch = batch; d->mb_row0 = row0;
    return;
  }
  const int64_t n_batches = ceil_div64(rows, batch);
  int64_t gb = n_batches;                              // resident data: one group
  if (d->cols_pending) {
    // one-shot path, columns and values still crossing PCIe: build group by group behind the upload
    const double per_batch = (double)d->nnz / (double)n_batches;
    const double group_entries = getenv("FMWR_GROUP_ENTRIES") ? atof(getenv("FMWR_GROUP_ENTRIES")) : (double)(32ll << 20);
    gb = std::min(n_batches, (int64_t)std::max(1.0, std::floor(group_entries / std::max(1.0, per_batch))));
  }
  const int gbits = bits_for((uint64_t)(gb - 1));
  const int bits = bits_for((uint64_t)(d->p > 0 ? d->p - 1 : 0)) + gbits;
  if (bits <= 32) minibatch_build_grouped<uint32_t>(d, row0, batch, gb, gbits);     // (batch, feature) fits one word: half the sort traffic
  else minibatch_build_grouped<uint64_t>(d, row0, batch, gb, gbits);
}

static void minibatch_fill_values(fmwr_data* d, uint32_t seg_lo, uint32_t seg_hi)
{
  if (seg_hi <= seg_lo) return;
  FMWR_LAUNCH(d->ctx, mb_fill_values, ceil_div((int64_t)seg_hi - seg_lo, 256), 256, 0, d->mb_seg_ptr.p, d->mb_seg_rec.p, d->mb_perm.p, d->val.p,
              d->mb_e0, seg_lo, seg_hi, d->mb_ent_val.p);
}

// the values of batch b of the per-batch CSC ready on the compute stream: it waits for the value chunks that hold the batch's
// entries, narrows the raw ones and fills the batch's segments (nothing to do once every value is in place)
void minibatch_batch_values(fmwr_data* d, int64_t b)
{
  if (!d->mb_vals_pending) return;
  const int64_t lo = b == 0 ? 0 : (int64_t)d->mb_e0 + d->mb_batch_ent[b], hi = (int64_t)d->mb_e0 + d->mb_batch_ent[b + 1];
  if (hi > 0) {
    const int64_t ci = std::min<int64_t>((int64_t)d->val_ev.size() - 1, (hi - 1) / d->val_chunk);
    data_wait_chunk_issued(d, ci);          // the event exists once the uploader has queued the chunk
    // every chunk up to ci (a mixed upload queues a raw chunk before the two narrowed ones in front of it)
    for (; d->val_waited <= ci; ++d->val_waited) FMWR_CUDA(cudaStreamWaitEvent(d->ctx->stream, d->val_ev[d->val_waited], 0));
  }
  data_narrow_values(d, lo, hi);
  minibatch_fill_values(d, (uint32_t)d->mb_batch_seg[b], (uint32_t)d->mb_batch_seg[b + 1]);
  if (b + 2 == (int64_t)d->mb_batch_seg.size()) { d->mb_vals_pending = false; d->val_all_narrowed = true; }     // the last batch
}

// every value of the per-batch CSC in place (a first epoch that stopped before its last batch)
void minibatch_all_values(fmwr_data* d)
{
  if (!d->mb_vals_pending) return;
  data_wait_values(d);
  minibatch_fill_values(d, 0u, (uint32_t)d->mb_batch_seg.back());
  d->mb_vals_pending = false;
}

int64_t minibatch_entries(const fmwr_data* d) { return d->mb_batch_ent.empty() ? 0 : d->mb_batch_ent.back(); }

// ------------------------------------------------------------------------------------------ scales / normalize
__global__ void col_moments(const uint32_t* __restrict__ col, const float* __restrict__ val, int64_t nnz,
                            double* __restrict__ sum, double* __restrict__ sumsq)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const double x = val[i];
  atomicAdd(sum + col[i], x);
  atomicAdd(sumsq + col[i], x * x);
}

__global__ void col_rescale(const uint32_t* __restrict__ col, float* __restrict__ val, int64_t nnz,
                            const double* __restrict__ mean, const double* __restrict__ sd, int mode)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t c = col[i];
  if (mode == 0) {
    // SMatrix::scales in-place step: float -= double; float /= (double + 1e-30)  (src/util/Smatrix.h:121-125)
    float x = val[i];
    x = (float)((double)x - mean[c]);
    x = (float)((double)x / (sd[c] + 1e-30));
    val[i] = x;
  } else {
    // SMatrix::normalize (src/util/Smatrix.h:144-150): skipped when std == 0
    if (sd[c] != 0) val[i] = (float)(((double)val[i] - mean[c]) / sd[c]);
  }
}

// A handle may outlive one call (the glue parks it inside the fm.matrix object, SURVEY 8f-3) and every fm.train / predict on it
// z-scores "the input": the passes below therefore always start from the values as uploaded.  The first pass keeps a
// pristine copy; later ones (and data_restore_values) copy it back first.
void data_values_from_raw(fmwr_data* d)
{
  data_wait_values(d);
  if (d->nnz == 0) return;
  if (!d->val_raw.p) {
    d->val_raw.alloc(d->nnz);
    FMWR_CUDA(cudaMemcpyAsync(d->val_raw.p, d->val.p, 4 * d->nnz, cudaMemcpyDeviceToDevice, d->ctx->stream));
  } else {
    FMWR_CUDA(cudaMemcpyAsync(d->val.p, d->val_raw.p, 4 * d->nnz, cudaMemcpyDeviceToDevice, d->ctx->stream));
  }
}

// undo a z-score pass (no-op on a handle that was never rescaled)
void data_restore_values(fmwr_data* d)
{
  if (!d->val_raw.p || d->nnz == 0) return;
  FMWR_CUDA(cudaMemcpyAsync(d->val.p, d->val_raw.p, 4 * d->nnz, cudaMemcpyDeviceToDevice, d->ctx->stream));
  d->val_raw.release();
  FMWR_CUDA(cudaStreamSynchronize(d->ctx->stream));
  d->has_csc = false; d->mb_batch = 0; d->als_cache.reset();   // derived layouts hold the rescaled values
}

void data_set_labels(fmwr_data* d, const double* labels) { set_labels_f64(d, labels); d->ctx->h2d_bytes += 8 * d->n; }

void data_scales(fmwr_data* d, const int32_t* norm_cols, int64_t n_norm, double* mean, double* sd)
{
  fmwr_ctx* ctx = d->ctx;
  const int64_t p = d->p, n = d->n;
  data_values_from_raw(d);
  DBuf<double> s, q;
  s.alloc(p); q.alloc(p);
  s.zero(ctx->stream); q.zero(ctx->stream);
  if (d->nnz > 0) FMWR_LAUNCH(ctx, col_moments, ceil_div(d->nnz, 256), 256, 0, d->col.p, d->val.p, d->nnz, s.p, q.p);
  std::vector<double> hs(p), hq(p);
  FMWR_CUDA(cudaMemcpyAsync(hs.data(), s.p, 8 * p, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(hq.data(), q.p, 8 * p, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  // per-column statistics exactly as src/util/Smatrix.h:111-119 (unlisted columns: mean 0, std 1)
  const double mult_dim = (double)n * ((double)n - 1);
  int64_t i = 0;
  for (int64_t c = 0; c < p; ++c) {
    if (i < n_norm && c == (int64_t)norm_cols[i]) {
      sd[c] = std::sqrt(hq[c] / (double)(uint32_t)(n - 1) - hs[c] * hs[c] / mult_dim);
      mean[c] = hs[c] / (double)n;
      ++i;
    } else { sd[c] = 1.0; mean[c] = 0.0; }
  }
  FMWR_CUDA(cudaMemcpyAsync(s.p, mean, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(q.p, sd, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
  if (d->nnz > 0) FMWR_LAUNCH(ctx, col_rescale, ceil_div(d->nnz, 256), 256, 0, d->col.p, d->val.p, d->nnz, s.p, q.p, 0);
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  d->has_csc = false; d->mb_batch = 0; d->als_cache.reset();   // derived layouts hold stale values
}

void data_normalize(fmwr_data* d, const double* mean, const double* sd)
{
  fmwr_ctx* ctx = d->ctx;
  const int64_t p = d->p;
  data_values_from_raw(d);
  DBuf<double> s, q;
  s.alloc(p); q.alloc(p);
  FMWR_CUDA(cudaMemcpyAsync(s.p, mean, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(q.p, sd, 8 * p, cudaMemcpyHostToDevice, ctx->stream));
  if (d->nnz > 0) FMWR_LAUNCH(ctx, col_rescale, ceil_div(d->nnz, 256), 256, 0, d->col.p, d->val.p, d->nnz, s.p, q.p, 1);
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  d->has_csc = false; d->mb_batch = 0; d->als_cache.reset();
}

// ------------------------------------------------------------------------------------------ synthetic data
// id(row, field) = offset_f + skewed(h(seed, row*F + field)) mod size_f          (SURVEY section 8d)
// h = splitmix64(seed ^ (row*F + field)); integer-only so the numpy twin (fmwr_b200/synth.py) is bit-identical.
__device__ __host__ __forceinline__ uint64_t synth_id(uint64_t h, uint64_t size, int skew)
{
  if (!skew) return h % size;
  // power-law skew: u^3 in 32.32 fixed point, then scaled to [0, size)
  const uint64_t u = h >> 32;                       // 32-bit uniform
  const uint64_t u2 = (u * u) >> 32;
  const uint64_t u3 = (u2 * u) >> 32;
  return (u3 * size) >> 32;
}

__device__ __host__ __forceinline__ float synth_value(uint64_t h, int value_mode)
{
  if (!value_mode) return 1.0f;
  // second hash word -> 24-bit mantissa, exactly representable: x in [0.5, 1.5)
  const uint64_t h2 = splitmix64(h ^ 0xD1B54A32D192ED03ull);
  return 0.5f + (float)(h2 >> 40) * (1.0f / 16777216.0f);
}

struct SynthFields {
  uint64_t offset[64];
  uint64_t size[64];
  int skew[64];
};

__global__ void synth_fill(int64_t n, int64_t row_begin, int F, SynthFields f, int value_mode, uint64_t seed,
                           uint32_t* __restrict__ rowptr, uint32_t* __restrict__ col, float* __restrict__ val)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // local entry index
  if (i <= n) { if (i * F <= 0xffffffffll) rowptr[i] = (uint32_t)(i * F); }
  if (i >= n * F) return;
  const int64_t row = i / F;
  const int fld = (int)(i - row * F);
  const uint64_t h = splitmix64(seed ^ (uint64_t)((row_begin + row) * F + fld));   // keyed by the GLOBAL entry index
  col[i] = (uint32_t)(f.offset[fld] + synth_id(h, f.size[fld], f.skew[fld]));
  val[i] = synth_value(h, value_mode);
}

// standard normal from two hash words (Box-Muller), double precision
__device__ __forceinline__ double hash_normal(uint64_t key)
{
  const uint64_t a = splitmix64(key), b = splitmix64(key ^ 0xA0761D6478BD642Full);
  const double u1 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  const double u2 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

template <class T>
__global__ void fill_normal(T* __restrict__ a, int64_t n, int k, int kp, double mean, double sd, uint64_t seed)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // index into the padded [p][kp] array
  if (i >= n) return;
  const int f = (int)(i % kp);
  const int64_t j = i / kp;
  a[i] = (f < k) ? T(mean + sd * hash_normal(seed ^ (uint64_t)(j * k + f))) : T(0);
}

template <class T>
__global__ void synth_labels(const T* __restrict__ score, int64_t n, int64_t row_begin, int label_mode, double noise, uint64_t seed,
                             float* __restrict__ y)
{
  const int64_t li = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n) return;
  const double s = (double)score[li];
  const int64_t i = row_begin + li;      // noise keyed by the global row
  if (label_mode == 1) {
    const double u = ((double)(splitmix64(seed ^ (uint64_t)i) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    y[li] = (u < 1.0 / (1.0 + exp(-s))) ? 1.0f : -1.0f;
  } else if (label_mode == 2) {
    y[li] = (float)(s + noise * hash_normal(seed ^ (uint64_t)i));
  } else {
    double t = 3.5 + s + noise * hash_normal(seed ^ (uint64_t)i);
    t = t < 0.5 ? 0.5 : (t > 5.0 ? 5.0 : t);
    y[li] = (float)t;
  }
}

__global__ void minmax_f32(const float* __restrict__ y, int64_t n, float* __restrict__ out /*[2]: -min, max as ordered ints*/)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float mn = INFINITY, mx = -INFINITY;
  if (i < n) { mn = y[i]; mx = y[i]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    // float atomic min/max through the sign-aware int trick
    int* o = (int*)out;
    if (mn >= 0) atomicMin(o, __float_as_int(mn)); else atomicMax((unsigned*)o, __float_as_uint(mn));
    if (mx >= 0) atomicMax(o + 1, __float_as_int(mx)); else atomicMin((unsigned*)(o + 1), __float_as_uint(mx));
  }
}

void model_init_random(fmwr_model* m, double mean, double sd, uint64_t seed)
{
  fmwr_ctx* ctx = m->ctx;
  const int64_t tot = m->p * m->kp;
  FMWR_CUDA(cudaMemsetAsync(m->scal.p, 0, m->scal.bytes(), ctx->stream));
  FMWR_CUDA(cudaMemsetAsync(m->w.p, 0, m->w.bytes(), ctx->stream));
  if (m->prec == FMWR_F64) FMWR_LAUNCH(ctx, fill_normal<double>, ceil_div(tot, 256), 256, 0, (double*)m->v.p, tot, m->k, m->kp, mean, sd, seed);
  else FMWR_LAUNCH(ctx, fill_normal<float>, ceil_div(tot, 256), 256, 0, (float*)m->v.p, tot, m->k, m->kp, mean, sd, seed);
}

void data_synth(fmwr_ctx* ctx, int64_t n, int64_t row_begin, int32_t n_fields, const int64_t* field_size, const int32_t* skew,
                int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out)
{
  FMWR_REQUIRE(n_fields > 0 && n_fields <= 64, FMWR_ERR_ARG, "n_fields must be in [1, 64]");
  SynthFields sf;
  uint64_t off = 0;
  for (int f = 0; f < n_fields; ++f) {
    FMWR_REQUIRE(field_size[f] > 0, FMWR_ERR_ARG, "field_size must be positive");
    sf.offset[f] = off; sf.size[f] = (uint64_t)field_size[f]; sf.skew[f] = skew ? skew[f] : 0;
    off += (uint64_t)field_size[f];
  }
  const int64_t p = (int64_t)off, nnz = n * n_fields;
  FMWR_REQUIRE(nnz < (int64_t)0xffffffffll && p < (int64_t)0xffffffffll, FMWR_ERR_UNSUPPORTED,
               "dimensions must fit 32-bit indices per device shard");
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = n; d->p = p; d->nnz = nnz;
    d->rowptr.alloc(n + 1); d->col.alloc(nnz); d->val.alloc(nnz);
    const int64_t threads = std::max(nnz, n + 1);
    FMWR_LAUNCH(ctx, synth_fill, ceil_div(threads, 256), 256, 0, n, row_begin, n_fields, sf, value_mode, seed, d->rowptr.p, d->col.p, d->val.p);
    if (label_mode != 0) {
      // planted FM (k* = 8, w*, V* ~ N(0, 0.1^2)) scored with the engine's own forward kernel
      fmwr_model_cfg mc; memset(&mc, 0, sizeof mc);
      mc.task = FMWR_REGRESSION; mc.keep_w0 = 1; mc.keep_w1 = 1; mc.k = 8;
      fmwr_model* pm = nullptr;
      FMWR_REQUIRE(fmwr_model_create(ctx, &mc, p, FMWR_F32, &pm) == 0, FMWR_ERR_CUDA, fmwr_last_error());
      try {
        model_init_random(pm, 0.0, 0.1, seed + 1);
        const int64_t pw = p;
        FMWR_LAUNCH(ctx, fill_normal<float>, ceil_div(pw, 256), 256, 0, (float*)pm->w.p, pw, 1, 1, 0.0, 0.1, seed + 2);
        forward_launch(ctx, pm, d, FMWR_LINK_NONE, 0, 0);
        d->y.alloc(n); d->has_labels = true;
        FMWR_LAUNCH(ctx, synth_labels<double>, ceil_div(n, 256), 256, 0, d->pred64.p, n, row_begin, label_mode, noise, seed + 3, d->y.p);
        DBuf<float> mm; mm.alloc(2);
        const float init[2] = {INFINITY, -INFINITY};
        FMWR_CUDA(cudaMemcpyAsync(mm.p, init, 8, cudaMemcpyHostToDevice, ctx->stream));
        FMWR_LAUNCH(ctx, minmax_f32, ceil_div(n, 256), 256, 0, d->y.p, n, mm.p);
        float h[2];
        FMWR_CUDA(cudaMemcpyAsync(h, mm.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
        FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
        d->min_y = h[0]; d->max_y = h[1];
      } catch (...) { fmwr_model_destroy(pm); throw; }
      fmwr_model_destroy(pm);
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } catch (...) { delete d; throw; }
  *out = d;
}

// ------------------------------------------------------------------------------------------ column slice
// rows keep only the entries with column in [c0, c1); ids are rebased to c - c0 (feature-parallel sharding)
__global__ void slice_count(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, int64_t n, uint32_t c0,
                            uint32_t c1, uint32_t* __restrict__ cnt, uint32_t* __restrict__ first)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t b = rowptr[r], e = rowptr[r + 1];
  uint32_t lo = b, hi = e;                        // first entry with col >= c0 (columns ascend inside a row)
  while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (col[m] < c0) lo = m + 1; else hi = m; }
  const uint32_t f = lo;
  hi = e;
  while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (col[m] < c1) lo = m + 1; else hi = m; }
  first[r] = f;
  cnt[r] = lo - f;
}

__global__ void slice_copy(const uint32_t* __restrict__ first, const uint32_t* __restrict__ new_rowptr, const uint32_t* __restrict__ col,
                           const float* __restrict__ val, int64_t n, uint32_t c0, uint32_t* __restrict__ ocol, float* __restrict__ oval)
{
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const uint32_t ob = new_rowptr[r], cnt = new_rowptr[r + 1] - ob, f = first[r];
  for (uint32_t j = threadIdx.x & 31; j < cnt; j += 32) { ocol[ob + j] = col[f + j] - c0; oval[ob + j] = val[f + j]; }
}

fmwr_data* data_slice_columns(fmwr_data* src, int64_t c0, int64_t c1)
{
  fmwr_ctx* ctx = src->ctx;
  FMWR_REQUIRE(0 <= c0 && c0 <= c1 && c1 <= src->p, FMWR_ERR_ARG, "column range out of bounds");
  const int64_t n = src->n;
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = n; d->p = c1 - c0;
    d->rowptr.alloc(n + 1);
    DBuf<uint32_t> cnt, first;
    cnt.alloc(n + 1); first.alloc(n + 1);
    FMWR_CUDA(cudaMemsetAsync(cnt.p, 0, 4 * (n + 1), ctx->stream));
    if (n > 0) FMWR_LAUNCH(ctx, slice_count, ceil_div(n, 256), 256, 0, src->rowptr.p, src->col.p, n, (uint32_t)c0, (uint32_t)c1, cnt.p, first.p);
    exclusive_scan_u32(ctx, cnt.p, d->rowptr.p, n + 1);
    uint32_t total = 0;
    FMWR_CUDA(cudaMemcpy(&total, d->rowptr.p + n, 4, cudaMemcpyDeviceToHost));
    d->nnz = total;
    d->col.alloc(total); d->val.alloc(total);
    if (n > 0 && total > 0) FMWR_LAUNCH(ctx, slice_copy, ceil_div(n * 32, 256), 256, 0, first.p, d->rowptr.p, src->col.p, src->val.p, n, (uint32_t)c0, d->col.p, d->val.p);
    if (src->has_labels) {
      d->y.alloc(n); d->has_labels = true; d->min_y = src->min_y; d->max_y = src->max_y;
      FMWR_CUDA(cudaMemcpyAsync(d->y.p, src->y.p, 4 * n, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } catch (...) { delete d; throw; }
  return d;
}

// ------------------------------------------------------------------------------------------ row gather
__global__ void gather_row_sizes(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ order, int64_t m, uint32_t* __restrict__ cnt)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) { const uint32_t r = order[i]; cnt[i] = rowptr[r + 1] - rowptr[r]; }
}
__global__ void gather_row_entries(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, const float* __restrict__ val, const float* __restrict__ y,
                                   const uint32_t* __restrict__ order, const uint32_t* __restrict__ new_rowptr, int64_t m,
                                   uint32_t* __restrict__ ocol, float* __restrict__ oval, float* __restrict__ oy)
{
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= m) return;
  const uint32_t r = order[i], b = rowptr[r], cnt = rowptr[r + 1] - b, ob = new_rowptr[i];
  for (uint32_t j = threadIdx.x & 31; j < cnt; j += 32) { ocol[ob + j] = col[b + j]; oval[ob + j] = val[b + j]; }
  if (oy && (threadIdx.x & 31) == 0) oy[i] = y[r];
}

// rows order[0], order[1], ... of src (repeats allowed) as a dataset of its own: how the throughput mode follows a strided
// visit sequence (random_step > 1) -- its batches are consecutive VISITS
fmwr_data* data_gather_rows(fmwr_data* src, const uint32_t* order_dev, int64_t m)
{
  fmwr_ctx* ctx = src->ctx;
  data_wait_cols(src);
  data_wait_values(src);
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = m; d->p = src->p;
    d->rowptr.alloc(m + 1);
    DBuf<uint32_t> cnt;
    cnt.alloc(m + 1);
    FMWR_CUDA(cudaMemsetAsync(cnt.p, 0, 4 * (m + 1), ctx->stream));
    if (m > 0) FMWR_LAUNCH(ctx, gather_row_sizes, ceil_div(m, 256), 256, 0, src->rowptr.p, order_dev, m, cnt.p);
    exclusive_scan_u32(ctx, cnt.p, d->rowptr.p, m + 1);
    uint32_t total = 0;
    FMWR_CUDA(cudaMemcpy(&total, d->rowptr.p + m, 4, cudaMemcpyDeviceToHost));
    d->nnz = total;
    d->col.alloc(total); d->val.alloc(total);
    if (src->has_labels) { d->y.alloc(m); d->has_labels = true; d->min_y = src->min_y; d->max_y = src->max_y; }
    if (m > 0) FMWR_LAUNCH(ctx, gather_row_entries, ceil_div(m * 32, 256), 256, 0, src->rowptr.p, src->col.p, src->val.p, src->has_labels ? src->y.p : nullptr,
                           order_dev, d->rowptr.p, m, d->col.p, d->val.p, src->has_labels ? d->y.p : nullptr);
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } catch (...) { delete d; throw; }
  return d;
}

// ------------------------------------------------------------------------------------------ row concatenation
__global__ void add_offset_u32(const uint32_t* __restrict__ in, int64_t n, uint32_t off, uint32_t* __restrict__ out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] + off;
}

// rows of parts[0], then parts[1], ...: how a shard too large to generate in one piece is assembled (bench.py builds the
// 100M-row column slices of BASELINE configs[4] from 10M-row chunks)
fmwr_data* data_concat_rows(fmwr_data* const* parts, int n_parts)
{
  FMWR_REQUIRE(n_parts > 0 && parts && parts[0], FMWR_ERR_ARG, "nothing to concatenate");
  fmwr_ctx* ctx = parts[0]->ctx;
  int64_t n = 0, nnz = 0;
  for (int i = 0; i < n_parts; ++i) {
    FMWR_REQUIRE(parts[i] && parts[i]->ctx == ctx && parts[i]->p == parts[0]->p && parts[i]->has_labels == parts[0]->has_labels, FMWR_ERR_SHAPE,
                 "parts must share context, feature count and label presence");
    n += parts[i]->n; nnz += parts[i]->nnz;
  }
  for (int i = 0; i < n_parts; ++i) { data_wait_cols(parts[i]); data_wait_values(parts[i]); }
  FMWR_REQUIRE(nnz < (int64_t)0xffffffffll && n < (int64_t)0xffffffffll, FMWR_ERR_UNSUPPORTED, "dimensions must fit 32-bit indices per device shard");
  fmwr_data* d = new fmwr_data();
  try {
    d->ctx = ctx; d->n = n; d->p = parts[0]->p; d->nnz = nnz; d->has_labels = parts[0]->has_labels;
    d->rowptr.alloc(n + 1); d->col.alloc(nnz); d->val.alloc(nnz);
    if (d->has_labels) d->y.alloc(n);
    d->min_y = INFINITY; d->max_y = -INFINITY;
    int64_t r0 = 0, e0 = 0;
    for (int i = 0; i < n_parts; ++i) {
      fmwr_data* q = parts[i];
      if (q->n > 0) FMWR_LAUNCH(ctx, add_offset_u32, ceil_div(q->n, 256), 256, 0, q->rowptr.p, q->n, (uint32_t)e0, d->rowptr.p + r0);
      if (q->nnz > 0) {
        FMWR_CUDA(cudaMemcpyAsync(d->col.p + e0, q->col.p, 4 * q->nnz, cudaMemcpyDeviceToDevice, ctx->stream));
        FMWR_CUDA(cudaMemcpyAsync(d->val.p + e0, q->val.p, 4 * q->nnz, cudaMemcpyDeviceToDevice, ctx->stream));
      }
      if (d->has_labels && q->n > 0) {
        FMWR_CUDA(cudaMemcpyAsync(d->y.p + r0, q->y.p, 4 * q->n, cudaMemcpyDeviceToDevice, ctx->stream));
        d->min_y = std::min(d->min_y, q->min_y); d->max_y = std::max(d->max_y, q->max_y);
      }
      r0 += q->n; e0 += q->nnz;
    }
    const uint32_t last = (uint32_t)nnz;
    FMWR_CUDA(cudaMemcpyAsync(d->rowptr.p + n, &last, 4, cudaMemcpyHostToDevice, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } catch (...) { delete d; throw; }
  return d;
}

}  // namespace fmwr
