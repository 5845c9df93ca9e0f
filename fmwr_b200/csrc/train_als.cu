// ALS / MCMC coordinate passes over the CSC twin.
//
// Replaces MCMC_ALS_Learner::{learn, update_all, calculate_error, update_alpha, update_w0, update_w,
// update_v, update_w_lambda, update_w_mu, update_v_lambda, update_v_mu}
// (reference src/solver/MCMC_ALS_Learner.h:91-562) at nthreads = 1, i.e. exact Gauss-Seidel in feature
// order.  GPU width comes from the "phase" decomposition (data.cu: phases_build): consecutive feature
// ranges whose members never share a row touch disjoint entries of the error vector e and of the
// per-row factor sums q, so updating them concurrently IS the sequential result.  For field-structured
// data (one-hot user/item/context, Criteo's 39 fields) a phase is a field.
//
// Per sweep (update_all order, :141-155): forward -> e (and q[r][f] = S_f of every row, which is what the
// reference rebuilds per factor at :286-299) -> calculate_error -> alpha -> w0 -> lambda_w -> mu_w -> w
// [-> lambda_v -> mu_v -> V when enable_v; the shipped code comments that block out, SURVEY F1].
// Hyper-parameters are the ones MCMC_ALS_Learner::init forces (alpha_0 = gamma_0 = beta_0 = 1, mu_0 = 0,
// alpha = 1, w0_mean_0 = 0; SURVEY F2), one attribute group (src/FM.cpp:75).
#include "forward.cuh"

#include <algorithm>
#include <cmath>
#include <random>

namespace fmwr {

template <class T> struct Vec2;
template <> struct Vec2<float> { typedef float2 type; };
template <> struct Vec2<double> { typedef double2 type; };

void comm_allreduce_sum(fmwr_ctx* ctx, void* buf, size_t count, bool f64);

// rows a warp contributes to a forward tile (tile = 8 warps x RW rows): as many as keep the staging buffer within 40 KB --
// longer runs of consecutive rows per factor in the transposed q stores (measured 1.9 -> 1.6 ms at k = 32 from 4 to 16)
template <class T, int KP, int TPW>
struct AlsTile {
  static constexpr int fit(int rw) { return (size_t)(KP + 1) * 8 * rw * sizeof(T) <= 40 * 1024; }
  static constexpr int BASE = fit(16) ? 16 : (fit(8) ? 8 : 4);
  static constexpr int RW = TPW > BASE ? TPW : BASE;
};
constexpr int ALS_LONG = 4096;      // columns at least this long get a whole CTA

// ---- forward: e = raw score, q[r][:] = S_f -----------------------------------------------------------
// A CTA (8 warps) works on tiles of TILE = 8 * RW rows, RW = max(4, rows per warp per pass).  q is factor-major
// [kp][n] (the coordinate passes stream one factor's q over rows), so the tile's S_f are staged in shared memory
// and every factor gets coalesced TILE-row stores.
template <class T, int LPR, int CH, int TEAM>
__global__ void __launch_bounds__(256, (LPR <= 8 && sizeof(T) == 4) ? 8 : 4)      // short rows: occupancy first (measured 2.4 -> 1.9 ms at k = 32)
als_forward_kernel(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
                   const T* __restrict__ w, const T* __restrict__ v, const double* __restrict__ scal, int kp, int k0, int k1,
                   int64_t n, T* __restrict__ e, T* __restrict__ q)
{
  constexpr int VN = Vec<T>::N;
  constexpr int KP = LPR * CH * VN;
  constexpr int TPW = 32 / TEAM;
  constexpr int RW = AlsTile<T, KP, TPW>::RW;
  constexpr int TILE = 8 * RW;
  constexpr bool STAGE = (size_t)(KP + 1) * TILE * sizeof(T) <= 40 * 1024;
  __shared__ T sS[STAGE ? TILE : 1][STAGE ? KP + 1 : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = lane / TEAM, tl = lane % TEAM;
  const T w0 = T(scal[0]);
  const int64_t n_tiles = (n + TILE - 1) / TILE;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row0 = tile * TILE;
#pragma unroll 1
    for (int i = 0; i < RW; i += TPW) {
      const int lr = warp * RW + i + team;
      const int64_t row = row0 + lr;
      uint32_t b = 0u, en = 0u;
      if (row < n) { b = __ldg(rowptr + row); en = __ldg(rowptr + row + 1); }
      T S[CH][VN];
      const T score = team_forward<T, LPR, CH, TEAM>(col, val, b, en, w, v, kp, w0, k0, k1, S);
      if (tl == 0 && row < n) e[row] = score;
      if (q && tl < LPR && row < n) {
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
#pragma unroll
          for (int j = 0; j < VN; ++j) {
            const int f = (ch * LPR + tl) * VN + j;
            if (STAGE) sS[lr][f] = S[ch][j];
            else q[(size_t)f * n + row] = S[ch][j];
          }
      }
    }
    if (STAGE && q) {
      __syncthreads();
      for (int f = warp; f < KP; f += 8)
#pragma unroll
        for (int r = lane; r < TILE; r += 32)
          if (row0 + r < n) q[(size_t)f * n + row0 + r] = sS[r][f];
      __syncthreads();
    }
  }
}

template <class T>
struct AlsFwd {
  fmwr_ctx* ctx; fmwr_model* m; fmwr_data* d; T* e; T* q; const uint32_t* col; const float* val;
  template <class TT, int LPR, int CH>
  void run()
  {
    if (short_rows(d->nnz, d->n, LPR)) go<TT, LPR, CH, LPR>();
    else go<TT, LPR, CH, 32>();
  }
  template <class TT, int LPR, int CH, int TEAM>
  void go()
  {
    constexpr int TPW = 32 / TEAM;
    constexpr int TILE = 8 * AlsTile<TT, LPR * CH * Vec<TT>::N, TPW>::RW;
    int64_t want = ceil_div64(d->n, TILE);
    int64_t cap = (int64_t)ctx->sm_count * 32;
    int grid = (int)std::max<int64_t>(1, std::min(want, cap));
    FMWR_LAUNCH(ctx, (als_forward_kernel<TT, LPR, CH, TEAM>), grid, 256, 0, d->rowptr.p, col, val, (const TT*)m->w.p,
                (const TT*)m->v.p, (const double*)m->scal.p, m->kp, m->cfg.keep_w0, m->cfg.keep_w1, d->n, e, q);
  }
};

// ---- uniform / normal sources ----------------------------------------------------------------------------
struct RandSrc {
  const int32_t* rands; long long n_rands;   // injected glibc rand() ints (NULL: counter hash)
  uint64_t seed;
};

__device__ __forceinline__ double hash_unif(uint64_t key)   // (0,1)
{
  return ((double)(splitmix64(key) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ double hash_norm(uint64_t key)
{
  const double u1 = hash_unif(key), u2 = hash_unif(key ^ 0xA0761D6478BD642Full);
  return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

// sequential uniform source: either the injected rand() stream (position in *pos) or a per-row counter hash
struct UnifStream {
  const int32_t* rands; long long n_rands; long long* pos; uint64_t key; uint32_t ctr;
  __device__ double next()
  {
    if (rands) {
      const long long i = (*pos)++;
      const int r = i < n_rands ? rands[i] : 0;
      return r / 2147483648.0;                                  // rand() / (RAND_MAX + 1), reference src/util/Random.h:20-24
    }
    return hash_unif(key + 0x9E3779B97F4A7C15ull * (++ctr));
  }
};

// fast_rnorm (Leva), reference src/util/Random.h:31-48
__device__ double leva_norm(UnifStream& s)
{
  double u, v, av, x, y, Q;
  do {
    do { u = s.next(); } while (u == 0.0);
    v = 1.7156 * (s.next() - 0.5);
    av = v < 0 ? -v : v;
    x = u - 0.449871;
    y = av + 0.386595;
    Q = x * x + y * (0.19600 * y - 0.25472 * x);
    if (Q < 0.27597) break;
  } while ((Q > 0.27846) || ((v * v) > (-4.0 * u * u * log(u))));
  return v / u;
}

// fast_trnorm_left(left) standard form, reference src/util/Random.h:51-76
__device__ double trnorm_left_std(UnifStream& s, double left)
{
  if (left < 0.0) {
    for (;;) { const double r = leva_norm(s); if (r >= left) return r; }
  }
  const double a = 0.5 * (left + sqrt(left * left + 4.0));
  for (;;) {
    const double z = -log(1 - s.next()) / a + left;
    double dd = z - a;
    dd = exp(-(dd * dd) / 2);
    const double u = s.next();
    if (u < dd) return z;
  }
}

// ---- calculate_error (reference :520-562) ------------------------------------------------------------------
// mode 0: regression e -= y; 1: ALS classification hazard table; 2: MCMC classification, truncated-normal draw
template <class T>
__global__ void als_error_kernel(T* __restrict__ e, const float* __restrict__ y, int64_t n, int mode,
                                 const double* __restrict__ dpY, uint64_t seed, uint64_t sweep, uint64_t row_offset)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double s = (double)e[i];
  const float yi = y[i];
  if (mode == 0) {
    e[i] = T(s - (double)yi);
  } else if (mode == 1) {
    e[i] = T(yi >= 0.0f ? -dev_fast_dpnorm(dpY, -s) : dev_fast_dpnorm(dpY, s));
  } else {
    UnifStream us{nullptr, 0, nullptr, splitmix64(seed ^ (sweep * 0xD6E8FEB86659FD93ull) ^ (row_offset + (uint64_t)i)), 0};
    // as shipped: N(0,1) truncated at the score (reference :536-539)
    const double t = yi >= 0.0f ? trnorm_left_std(us, s) : -trnorm_left_std(us, -s);
    e[i] = T(s - t);
  }
}

// injected rand() stream: rows consume a variable number of draws in row order -> one thread, validation sizes only
template <class T>
__global__ void als_error_stream_kernel(T* __restrict__ e, const float* __restrict__ y, int64_t n,
                                        const int32_t* __restrict__ rands, long long n_rands, long long* __restrict__ pos)
{
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  UnifStream us{rands, n_rands, pos, 0, 0};
  for (int64_t i = 0; i < n; ++i) {
    const double s = (double)e[i];
    const double t = y[i] >= 0.0f ? trnorm_left_std(us, s) : -trnorm_left_std(us, -s);
    e[i] = T(s - t);
  }
}

// ---- posterior mean (fmwr_train_posterior_dev) -------------------------------------------------------------------------
// One draw: acc[i] += link(score[i]) in f64, launched once per draw in draw order.  A kernel of its own rather than an
// accumulating variant of the error kernels: the eval sets need the same step on their forward results, and the kernels
// that drive the chain stay exactly as they are.  On the training rows it costs 4 bytes more per row (the score is read
// again) than a fused variant would, against ~146 GB of coordinate-pass traffic per sweep on the benchmark shape.
template <class S>
__global__ void posterior_accum_kernel(const S* __restrict__ score, int64_t n, int link, double lo, double hi,
                                       const double* __restrict__ pnY, double* __restrict__ acc)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) acc[i] += apply_link(link, (double)score[i], lo, hi, pnY);
}

// out[perm[i]] = acc[i] / draws (perm == nullptr: out[i]); a division, so that a host summing the same predictions in the
// same order gets the same bits
__global__ void posterior_mean_kernel(const double* __restrict__ acc, int64_t n, double draws, const uint32_t* __restrict__ perm,
                                      double* __restrict__ out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[perm ? (int64_t)perm[i] : i] = acc[i] / draws;
}

// ---- reductions ------------------------------------------------------------------------------------------
// mode 0: sum x, 1: sum x^2, 2: sum (x - c)^2
template <class T>
__global__ void als_reduce_kernel(const T* __restrict__ x, int64_t n, int64_t stride, int mode, double c, double* __restrict__ part)
{
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = (double)x[i * stride];
    acc += mode == 0 ? v : (mode == 1 ? v * v : (v - c) * (v - c));
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
    part[blockIdx.x] = s;
  }
}

// all factors at once: part[blk][f] = sum_c V[c][f], part[blk][kp + f] = sum_c (V[c][f] - mu[f])^2 over the block's
// columns.  One launch and one host round trip replace 2k of them in the MCMC hyper-prior step; the block partials are
// summed on the host in block order, so the result is deterministic.
template <class T>
__global__ void __launch_bounds__(256) als_reduce_v_kernel(const T* __restrict__ v, int64_t p, int kp, const double* __restrict__ mu,
                                                           int64_t cols_per_block, double* __restrict__ part)
{
  __shared__ double s1[256], s2[256];
  const int lanes_f = kp < 256 ? kp : 256;
  const int rows_par = 256 / lanes_f;
  const int my_f0 = threadIdx.x % lanes_f, my_r = threadIdx.x / lanes_f;
  const int64_t c0 = (int64_t)blockIdx.x * cols_per_block, c1 = c0 + cols_per_block < p ? c0 + cols_per_block : p;
  for (int fo = 0; fo < kp; fo += lanes_f) {
    const int f = fo + my_f0;
    double a1 = 0.0, a2 = 0.0;
    if (f < kp && my_r < rows_par) {
      const double m = mu[f];
      for (int64_t c = c0 + my_r; c < c1; c += rows_par) {
        const double x = (double)v[c * kp + f];
        a1 += x; a2 += (x - m) * (x - m);
      }
    }
    s1[threadIdx.x] = a1; s2[threadIdx.x] = a2;
    __syncthreads();
    if (my_r == 0 && f < kp) {
      for (int r = 1; r < rows_par; ++r) { a1 += s1[r * lanes_f + my_f0]; a2 += s2[r * lanes_f + my_f0]; }
      part[(size_t)blockIdx.x * 2 * kp + f] = a1;
      part[(size_t)blockIdx.x * 2 * kp + kp + f] = a2;
    }
    __syncthreads();
  }
}

// sums[f] = sum_c V[c][f], sq[f] = sum_c (V[c][f] - mu[f])^2, row0[f] = V[0][f]
template <class T>
static void reduce_v_all(fmwr_ctx* ctx, const T* v, int64_t p, int k, int kp, const std::vector<double>& mu, std::vector<double>& sums,
                         std::vector<double>& sq, std::vector<double>& row0)
{
  sums.assign(k, 0.0); sq.assign(k, 0.0); row0.assign(k, 0.0);
  if (p <= 0 || k <= 0) return;
  const int nblk = (int)std::min<int64_t>(256, std::max<int64_t>(1, ceil_div64(p, 512)));
  const int64_t cpb = ceil_div64(p, nblk);
  DBuf<double> mu_dev, part;
  mu_dev.alloc(kp); part.alloc((size_t)nblk * 2 * kp);
  std::vector<double> hm(kp, 0.0);
  for (int f = 0; f < k; ++f) hm[f] = mu[f];
  FMWR_CUDA(cudaMemcpyAsync(mu_dev.p, hm.data(), 8 * kp, cudaMemcpyHostToDevice, ctx->stream));
  FMWR_LAUNCH(ctx, als_reduce_v_kernel<T>, nblk, 256, 0, v, p, kp, mu_dev.p, cpb, part.p);
  std::vector<double> h((size_t)nblk * 2 * kp);
  std::vector<T> r0(kp);
  FMWR_CUDA(cudaMemcpyAsync(h.data(), part.p, 8 * h.size(), cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(r0.data(), v, sizeof(T) * kp, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int b = 0; b < nblk; ++b)
    for (int f = 0; f < k; ++f) { sums[f] += h[(size_t)b * 2 * kp + f]; sq[f] += h[(size_t)b * 2 * kp + kp + f]; }
  for (int f = 0; f < k; ++f) row0[f] = (double)r0[f];
}

template <class T>
static double reduce(fmwr_ctx* ctx, const T* x, int64_t n, int64_t stride, int mode, double c)
{
  if (n <= 0) return 0.0;
  const int nblk = (int)std::min<int64_t>(1024, std::max<int64_t>(1, ceil_div64(n, 256)));
  ctx->red_scratch.ensure(1024);
  FMWR_LAUNCH(ctx, als_reduce_kernel<T>, nblk, 256, 0, x, n, stride, mode, c, ctx->red_scratch.p);
  std::vector<double> h(nblk);
  FMWR_CUDA(cudaMemcpyAsync(h.data(), ctx->red_scratch.p, 8 * nblk, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  double s = 0;
  for (int i = 0; i < nblk; ++i) s += h[i];
  return s;
}

template <class T>
__global__ void als_shift_kernel(T* __restrict__ e, int64_t n, T d)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) e[i] -= d;
}

// ---- coordinate kernels --------------------------------------------------------------------------------
template <class T>
struct CoordArgs {
  const uint32_t* colptr; const uint32_t* crow; const float* cval;
  uint32_t c_begin, c_end;           // the phase's feature range
  const uint32_t* long_cols; int n_long;
  T* e; T* q; int kp; int f; int64_t n;   // q == nullptr for the w pass; q is [kp][n]
  T* theta; int64_t theta_stride;    // w (stride 1) or V + f (stride kp)
  double alpha, lambda, mu;
  int do_sample; int w_sd_is_var;    // F7: w drawn with the variance as s.d.
  const double* normals; long long n_normals; long long normal_base;   // draw for column c: normals[normal_base + c]
  uint64_t seed;
};

template <class T>
__device__ __forceinline__ bool dev_bad(T x) { return isnan(x) || isinf(x); }

// one feature; `part` = number of cooperating threads, `tid` = index inside the group; reduce() sums over the group
template <class T, class Reduce>
__device__ __forceinline__ void coord_update(const CoordArgs<T>& a, uint32_t c, int tid, int part, Reduce reduce)
{
  const uint32_t b = a.colptr[c], en = a.colptr[c + 1];
  T* th = a.theta + (size_t)c * a.theta_stride;
  const double old = (double)*th;
  double A = 0.0, Bm = 0.0;
  if (a.q == nullptr) {
    // update_w statistics (reference :225-230): A = sum x^2, Bm = sum (e x - w x^2)
    for (uint32_t j = b + tid; j < en; j += part) {
      const double x = (double)a.cval[j];
      Bm += (double)a.e[a.crow[j]] * x - old * x * x;
      A += x * x;
    }
  } else {
    // update_v statistics (reference :313-321): h = x q - x^2 v, A = sum h^2, Bm = sum h e
    for (uint32_t j = b + tid; j < en; j += part) {
      const float xf = a.cval[j];
      const uint32_t r = a.crow[j];
      const double h = (double)xf * (double)a.q[(size_t)a.f * a.n + r] - (double)(xf * xf) * old;
      Bm += h * (double)a.e[r];
      A += h * h;
    }
  }
  A = reduce(A);
  Bm = reduce(Bm);
  if (a.q != nullptr) Bm -= old * A;                                   // :322
  const double var = 1.0 / (a.lambda + a.alpha * A);
  const double mean = -var * (a.alpha * Bm - a.mu * a.lambda);
  double nv;
  bool upd = true;
  if (dev_bad(var)) nv = 0.0;                                           // :235-236, :326-327
  else if (a.do_sample) {
    const long long di = a.normal_base + (long long)c;
    const double z = a.normals ? (di < a.n_normals ? a.normals[di] : 0.0) : hash_norm(a.seed ^ (uint64_t)di * 0x9E3779B97F4A7C15ull);
    const double sd = (a.q == nullptr && a.w_sd_is_var) ? var : sqrt(var);   // :239 (F7) vs :330
    nv = mean + sd * z;
  } else nv = mean;
  if (dev_bad(nv)) { nv = old; upd = false; }                           // CHECK_PARAM
  if (tid == 0) *th = T(nv);
  if (!upd) return;
  const double dlt = old - nv;
  if (a.q == nullptr) {
    for (uint32_t j = b + tid; j < en; j += part) {
      const uint32_t r = a.crow[j];
      a.e[r] = T((double)a.e[r] - (double)a.cval[j] * dlt);             // :251-253
    }
  } else {
    for (uint32_t j = b + tid; j < en; j += part) {
      const float xf = a.cval[j];
      const uint32_t r = a.crow[j];
      const size_t qi = (size_t)a.f * a.n + r;
      const double qv = (double)a.q[qi];
      const double h = (double)xf * qv - (double)(xf * xf) * old;
      a.q[qi] = T(qv - (double)xf * dlt);                               // :346
      a.e[r] = T((double)a.e[r] - h * dlt);                             // :347
    }
  }
}

// warp per feature (short columns); long ones are left to the CTA kernel
template <class T>
__global__ void __launch_bounds__(256) coord_warp_kernel(CoordArgs<T> a)
{
  const uint32_t c = a.c_begin + (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
  if (c >= a.c_end) return;
  const uint32_t len = a.colptr[c + 1] - a.colptr[c];
  if (len >= ALS_LONG) return;
  coord_update<T>(a, c, threadIdx.x & 31, 32, [](double v) { return warp_sum(v); });
}

template <class T>
__global__ void __launch_bounds__(512) coord_block_kernel(CoordArgs<T> a)
{
  __shared__ double red[16];
  __shared__ double tot;
  const uint32_t c = a.long_cols[blockIdx.x];
  auto block_sum = [&](double v) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0;
      for (int i = 0; i < 16; ++i) s += red[i];
      tot = s;
    }
    __syncthreads();
    return tot;
  };
  coord_update<T>(a, c, threadIdx.x, 512, block_sum);
}


// ---- row-major (streaming) coordinate passes ---------------------------------------------------------------
// Inside a phase every row holds at most one of the phase's features, so the phase's non-zeros can be visited in ROW
// order: e[r] and q[f][r] are then read and written as coalesced streams instead of 4-byte random gathers (which move a
// 32-byte sector each).  Per (factor, phase):
//   rm_extract   th[c]   <- current parameter of every feature of the phase (compact copy, L2-resident)
//   rm_stats     A[c], B[c] <- sum h^2, sum h e   (w pass: sum x^2, sum (e x - w x^2)); warp-aggregated vector atomics,
//                            shared-memory privatisation when the phase has few features
//   rm_solve     new parameter per feature (ALS mean / MCMC draw, the reference's NaN/Inf guards), delta[c] = old - new
//   rm_apply     e[r] -= h delta, q[f][r] -= x delta
// The phase's non-zeros are stored once, grouped by phase in row order (build_row_major).
struct RowMajor {
  bool ok = false;
  DBuf<uint32_t> row, col;      // [N] row id, feature id LOCAL to its phase
  DBuf<float> val;              // [N]
  std::vector<int64_t> ptr;     // [n_phases + 1] entry offsets
  uint32_t max_cols = 0;
  DBuf<uint32_t> hot_col;       // [n_phases][RM_HOT] phase-local feature id of each hot slot
  DBuf<uint16_t> hot;           // [p] slot of a hot feature inside its phase's shared-memory table, 0xffff otherwise
  std::vector<int> n_hot;       // [n_phases]
};

__global__ void rm_phase_keys(const uint32_t* __restrict__ col, int64_t nnz, const uint32_t* __restrict__ pbeg, int n_phases,
                              uint32_t* __restrict__ key)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t c = col[i];
  int lo = 0, hi = n_phases;                       // last phase with begin <= c
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pbeg[mid] <= c) lo = mid; else hi = mid; }
  key[i] = (uint32_t)lo;
}

__global__ void rm_emit(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ key_sorted, const uint32_t* __restrict__ erow,
                        const uint32_t* __restrict__ col, const float* __restrict__ val, const uint32_t* __restrict__ pbeg, int64_t nnz,
                        uint32_t* __restrict__ orow, uint32_t* __restrict__ ocol, float* __restrict__ oval)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t e = perm[i];
  orow[i] = erow[e];
  ocol[i] = col[e] - pbeg[key_sorted[i]];
  oval[i] = val[e];
}

__global__ void rm_expand_rows(const uint32_t* __restrict__ rowptr, int64_t n, uint32_t* __restrict__ erow)
{
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const uint32_t b = rowptr[row], e = rowptr[row + 1];
  for (uint32_t j = b + (threadIdx.x & 31); j < e; j += 32) erow[j] = (uint32_t)row;
}

__global__ void rm_count_phase(const uint32_t* __restrict__ key_sorted, int64_t nnz, int n_phases, unsigned long long* __restrict__ first)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t k = key_sorted[i];
  if (i == 0 || key_sorted[i - 1] != k) first[k] = (unsigned long long)i;
  (void)n_phases;
}

template <class T>
struct RmArgs {
  const uint32_t* row; const uint32_t* col; const float* val;
  int64_t pb, pe;                    // entry range of the phase
  uint32_t cb, ncols;                // first global feature / number of features of the phase
  T* e; T* q; int64_t n; int f;      // q == nullptr: w pass.  q is [kp][n]
  T* theta; int64_t theta_stride;    // w (stride 1) or V + f (stride kp)
  const uint16_t* hot; const uint32_t* hot_col; int n_hot;   // hot-feature table of the phase (indexed by global feature id)
  T* th; T* AB; T* delta;            // per-feature scratch of the phase: th[ncols], AB[n_rep][2*ncols] interleaved, delta[ncols]
  typename Vec2<T>::type* thd;       // (th, delta) interleaved: the fused passes fetch both with one gather (may be null)
  int n_rep;                         // replicas of the AB table (0/1: one); the fused passes spread their reductions over them
  size_t rep_stride;                 // distance between replicas in (A, B) pairs; 0: ncols (packed)
  double alpha, lambda, mu;
  int do_sample, w_sd_is_var;
  const double* normals; long long n_normals, normal_base; uint64_t seed;
};

template <class T> __device__ __forceinline__ void rm_extract_one(const RmArgs<T>& a, uint32_t c);
template <class T> __device__ __forceinline__ void rm_solve_one(const RmArgs<T>& a, uint32_t c);
template <class T> __device__ __forceinline__ void rm_solve_finish(const RmArgs<T>& a, uint32_t c, double A, double Bm);

template <class T>
__global__ void rm_extract_kernel(RmArgs<T> a)
{
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < a.ncols) rm_extract_one(a, c);
}

template <class T>
__global__ void rm_solve_kernel(RmArgs<T> a, PeerArgs pa, int peer)
{
  if (peer) peer_wait(pa, PEER_FLAG1, PEER_EPOCH1);        // row-sharded: every rank's statistics have arrived in our window
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < a.ncols) rm_solve_one(a, c);
}

// solve of step t and extract of step t + 1 in one launch (they touch different features and different scratch)
// 64 features x 4 replica slices per CTA: the replica sums / clears are latency chains, so they are spread over threads
constexpr int SE_COLS = 64, SE_SLICES = 4;
template <class T>
__global__ void __launch_bounds__(SE_COLS * SE_SLICES) rm_solve_extract_kernel(RmArgs<T> a, RmArgs<T> b, PeerArgs pa, int peer)
{
  typedef typename Vec2<T>::type V2;
  __shared__ double sA[SE_SLICES][SE_COLS], sB[SE_SLICES][SE_COLS];
  if (peer) peer_wait(pa, PEER_FLAG1, PEER_EPOCH1);        // row-sharded: every rank's statistics have arrived in our window
  const int tx = threadIdx.x % SE_COLS, ty = threadIdx.x / SE_COLS;
  const uint32_t c = blockIdx.x * SE_COLS + tx;
  double A = 0.0, Bm = 0.0;
  if (c < a.ncols) {
    const int R = a.n_rep > 1 ? a.n_rep : 1;
#pragma unroll 4
    for (int r = ty; r < R; r += SE_SLICES) {
      const V2 ab = reinterpret_cast<const V2*>(a.AB)[(size_t)r * (a.rep_stride ? a.rep_stride : a.ncols) + c];
      A += (double)ab.x; Bm += (double)ab.y;
    }
  }
  sA[ty][tx] = A; sB[ty][tx] = Bm;
  __syncthreads();
  if (ty == 0 && c < a.ncols) {
#pragma unroll
    for (int j = 1; j < SE_SLICES; ++j) { A += sA[j][tx]; Bm += sB[j][tx]; }
    rm_solve_finish(a, c, A, Bm);
  }
  if (c < b.ncols) {
    if (ty == 0) {
      const T th = b.theta[(size_t)(b.cb + c) * b.theta_stride];
      b.th[c] = th;
      if (b.thd) b.thd[c].x = th;
    }
    const int R = b.n_rep > 1 ? b.n_rep : 1;
    V2 z; z.x = T(0); z.y = T(0);
    for (int r = ty; r < R; r += SE_SLICES) reinterpret_cast<V2*>(b.AB)[(size_t)r * b.ncols + c] = z;
  }
}

template <class T>
__device__ __forceinline__ void rm_extract_one(const RmArgs<T>& a, uint32_t c)
{
  const T th = a.theta[(size_t)(a.cb + c) * a.theta_stride];
  a.th[c] = th;
  if (a.thd) a.thd[c].x = th;
  const int R = a.n_rep > 1 ? a.n_rep : 1;
  for (int r = 0; r < R; ++r) { a.AB[2 * ((size_t)r * a.ncols + c)] = T(0); a.AB[2 * ((size_t)r * a.ncols + c) + 1] = T(0); }
}

// A and B of a feature are interleaved (AB[2c], AB[2c+1]) so the fp32 path issues ONE 8-byte vector reduction per feature
__device__ __forceinline__ void atomic_add2(float* AB, uint32_t c, float a, float b)
{
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(AB + 2 * (size_t)c), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void atomic_add2(double* AB, uint32_t c, double a, double b) { atomicAdd(AB + 2 * (size_t)c, a); atomicAdd(AB + 2 * (size_t)c + 1, b); }

constexpr int RM_SMEM_COLS = 2048;

constexpr int RM_HOT = 4096;        // hot features per phase kept in a per-CTA shared-memory table
constexpr int RM_HOT_MIN_LEN = 512;   // a feature is hot when it has at least this many non-zeros

// MODE 0: global vector atomics (warp-aggregated); 1: the whole phase fits the shared-memory table;
// 2: hot features go to the shared-memory table, the rest to global atomics
template <class T, int MODE>
__global__ void __launch_bounds__(256) rm_stats_kernel(RmArgs<T> a)
{
  constexpr int HOT_SLOTS = sizeof(T) == 8 ? RM_HOT / 2 : RM_HOT;   // 32 KB of shared memory either way
  constexpr int SLOTS = MODE == 1 ? RM_SMEM_COLS : (MODE == 2 ? HOT_SLOTS : 1);
  __shared__ T sA[SLOTS], sB[SLOTS];
  const uint32_t n_slots = MODE == 1 ? a.ncols : (MODE == 2 ? (uint32_t)(a.n_hot < HOT_SLOTS ? a.n_hot : HOT_SLOTS) : 0u);
  if (MODE != 0) {
    for (uint32_t c = threadIdx.x; c < n_slots; c += blockDim.x) { sA[c] = T(0); sB[c] = T(0); }
    __syncthreads();
  }
  const T* qf = a.q ? a.q + (size_t)a.f * a.n : nullptr;
  for (int64_t i = a.pb + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.pe; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t r = a.row[i], c = a.col[i];
    const float xf = a.val[i];
    const T old = a.th[c];
    const T er = a.e[r];
    T sa, sb;
    if (qf == nullptr) {                          // update_w statistics (reference :225-230)
      const T x = T(xf);
      sa = x * x;
      sb = er * x - old * x * x;
    } else {                                      // update_v statistics (reference :313-321)
      const T h = T(xf) * qf[r] - T(xf * xf) * old;
      sa = h * h;
      sb = h * er;
    }
    if (MODE == 1) { atomicAdd(&sA[c], sa); atomicAdd(&sB[c], sb); continue; }
    if (MODE == 2) {
      const uint32_t slot = a.hot[a.cb + c];
      if (slot < n_slots) { atomicAdd(&sA[slot], sa); atomicAdd(&sB[slot], sb); continue; }
    }
    atomic_add2(a.AB, c, sa, sb);
  }
  if (MODE != 0) {
    __syncthreads();
    for (uint32_t sl = threadIdx.x; sl < n_slots; sl += blockDim.x)
      if (sA[sl] != T(0) || sB[sl] != T(0)) {
        const uint32_t c = MODE == 1 ? sl : a.hot_col[sl];
        atomic_add2(a.AB, c, sA[sl], sB[sl]);
      }
  }
}

template <class T>
__device__ __forceinline__ void rm_solve_one(const RmArgs<T>& a, uint32_t c)
{
  const double old = (double)a.th[c];
  double A = 0.0, Bm = 0.0;
  {
    const int R = a.n_rep > 1 ? a.n_rep : 1;
    typedef typename Vec2<T>::type V2;
#pragma unroll 8
    for (int r = 0; r < R; ++r) {
      const V2 ab = reinterpret_cast<const V2*>(a.AB)[(size_t)r * (a.rep_stride ? a.rep_stride : a.ncols) + c];
      A += (double)ab.x; Bm += (double)ab.y;
    }
  }
  rm_solve_finish(a, c, A, Bm);
}

template <class T>
__device__ __forceinline__ void rm_solve_finish(const RmArgs<T>& a, uint32_t c, double A, double Bm)
{
  const double old = (double)a.th[c];
  if (a.q != nullptr) Bm -= old * A;                                    // reference :322
  const double var = 1.0 / (a.lambda + a.alpha * A);
  const double mean = -var * (a.alpha * Bm - a.mu * a.lambda);
  double nv;
  bool upd = true;
  if (isnan(var) || isinf(var)) nv = 0.0;
  else if (a.do_sample) {
    const long long di = a.normal_base + (long long)(a.cb + c);
    const double z = a.normals ? (di < a.n_normals ? a.normals[di] : 0.0) : hash_norm(a.seed ^ (uint64_t)di * 0x9E3779B97F4A7C15ull);
    const double sd = (a.q == nullptr && a.w_sd_is_var) ? var : sqrt(var);
    nv = mean + sd * z;
  } else nv = mean;
  if (isnan(nv) || isinf(nv)) { nv = old; upd = false; }
  a.theta[(size_t)(a.cb + c) * a.theta_stride] = T(nv);
  a.delta[c] = upd ? T(old - nv) : T(0);
  if (a.thd) a.thd[c].y = upd ? T(old - nv) : T(0);
}

template <class T>
__global__ void __launch_bounds__(256) rm_apply_kernel(RmArgs<T> a)
{
  T* qf = a.q ? a.q + (size_t)a.f * a.n : nullptr;
  for (int64_t i = a.pb + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.pe; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t r = a.row[i], c = a.col[i];
    const T d = a.delta[c];
    if (d == T(0)) continue;
    const float xf = a.val[i];
    if (qf == nullptr) {
      a.e[r] -= T(xf) * d;                                              // reference :251-253
    } else {
      const T qv = qf[r];
      const T h = T(xf) * qv - T(xf * xf) * a.th[c];
      qf[r] = qv - T(xf) * d;                                           // :346
      a.e[r] -= h * d;                                                  // :347
    }
  }
}

static void build_row_major(fmwr_data* d, const std::vector<uint32_t>& pbeg_host, const std::vector<uint32_t>& cp, RowMajor& rm)
{
  fmwr_ctx* ctx = d->ctx;
  const int np = (int)pbeg_host.size() - 1;
  const int64_t nnz = d->nnz, n = d->n;
  rm.ptr.assign(np + 1, 0);
  rm.max_cols = 0;
  for (int i = 0; i < np; ++i) rm.max_cols = std::max(rm.max_cols, pbeg_host[i + 1] - pbeg_host[i]);
  if (nnz == 0) { rm.ok = true; return; }
  DBuf<uint32_t> pbeg, key_in, key_out, idx_in, idx_out, erow;
  DBuf<unsigned long long> first;
  pbeg.alloc(np + 1); key_in.alloc(nnz); key_out.alloc(nnz); idx_in.alloc(nnz); idx_out.alloc(nnz); erow.alloc(nnz); first.alloc(np + 1);
  FMWR_CUDA(cudaMemcpyAsync(pbeg.p, pbeg_host.data(), 4 * (np + 1), cudaMemcpyHostToDevice, ctx->stream));
  FMWR_LAUNCH(ctx, rm_phase_keys, ceil_div(nnz, 256), 256, 0, d->col.p, nnz, pbeg.p, np, key_in.p);
  FMWR_LAUNCH(ctx, rm_expand_rows, ceil_div(n * 32, 256), 256, 0, d->rowptr.p, n, erow.p);
  FMWR_CUDA(cudaMemsetAsync(first.p, 0xff, 8 * (np + 1), ctx->stream));
  // stable sort of entry ids by phase id: CSR order (== row order) survives inside each phase
  launch_iota(ctx, idx_in.p, nnz);
  int bits = 1;
  while ((1 << bits) < np) ++bits;
  sort_pairs_u32(ctx, key_in.p, key_out.p, idx_in.p, idx_out.p, nnz, bits);
  rm.row.alloc(nnz); rm.col.alloc(nnz); rm.val.alloc(nnz);
  FMWR_LAUNCH(ctx, rm_emit, ceil_div(nnz, 256), 256, 0, idx_out.p, key_out.p, erow.p, d->col.p, d->val.p, pbeg.p, nnz, rm.row.p, rm.col.p, rm.val.p);
  FMWR_LAUNCH(ctx, rm_count_phase, ceil_div(nnz, 256), 256, 0, key_out.p, nnz, np, first.p);
  std::vector<unsigned long long> hf(np + 1);
  FMWR_CUDA(cudaMemcpyAsync(hf.data(), first.p, 8 * (np + 1), cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  rm.ptr[np] = nnz;
  for (int i = np - 1; i >= 0; --i) rm.ptr[i] = (hf[i] == ~0ull) ? rm.ptr[i + 1] : (int64_t)hf[i];   // empty phase: zero-length range
  // hot features: the RM_HOT longest columns of every phase with at least RM_HOT_MIN_LEN non-zeros
  std::vector<uint16_t> hot(d->p > 0 ? d->p : 1, 0xffff);
  std::vector<uint32_t> hot_col((size_t)np * RM_HOT, 0);
  rm.n_hot.assign(np, 0);
  for (int i = 0; i < np; ++i) {
    std::vector<std::pair<uint32_t, uint32_t>> cand;     // (length, feature)
    for (uint32_t c = pbeg_host[i]; c < pbeg_host[i + 1]; ++c) {
      const uint32_t len = cp[c + 1] - cp[c];
      if (len >= (uint32_t)RM_HOT_MIN_LEN) cand.push_back({len, c});
    }
    if ((int)cand.size() > RM_HOT) {
      std::partial_sort(cand.begin(), cand.begin() + RM_HOT, cand.end(), [](const std::pair<uint32_t, uint32_t>& x, const std::pair<uint32_t, uint32_t>& y) { return x.first > y.first; });
      cand.resize(RM_HOT);
    }
    rm.n_hot[i] = (int)cand.size();
    for (size_t s2 = 0; s2 < cand.size(); ++s2) { hot[cand[s2].second] = (uint16_t)s2; hot_col[(size_t)i * RM_HOT + s2] = cand[s2].second - pbeg_host[i]; }
  }
  rm.hot.alloc(hot.size()); rm.hot_col.alloc(hot_col.size() ? hot_col.size() : 1);
  FMWR_CUDA(cudaMemcpyAsync(rm.hot.p, hot.data(), 2 * hot.size(), cudaMemcpyHostToDevice, ctx->stream));
  if (!hot_col.empty()) FMWR_CUDA(cudaMemcpyAsync(rm.hot_col.p, hot_col.data(), 4 * hot_col.size(), cudaMemcpyHostToDevice, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  rm.ok = true;
}

template <class T>
static void run_phases_rm(fmwr_ctx* ctx, const std::vector<uint32_t>& pbeg, const RowMajor& rm, RmArgs<T> a)
{
  const int np = (int)pbeg.size() - 1;
  const int grid_stream = ctx->sm_count * 8;
  for (int i = 0; i < np; ++i) {
    a.pb = rm.ptr[i]; a.pe = rm.ptr[i + 1];
    a.cb = pbeg[i]; a.ncols = pbeg[i + 1] - pbeg[i];
    if (a.ncols == 0) continue;
    FMWR_LAUNCH(ctx, rm_extract_kernel<T>, ceil_div(a.ncols, 256), 256, 0, a);
    if (a.pe > a.pb) {
      const int grid = (int)std::min<int64_t>(grid_stream, ceil_div64(a.pe - a.pb, 256));
      a.n_hot = rm.n_hot[i];
      a.hot_col = rm.hot_col.p + (size_t)i * RM_HOT;
      if (a.ncols <= RM_SMEM_COLS) FMWR_LAUNCH(ctx, (rm_stats_kernel<T, 1>), grid, 256, 0, a);
      else if (a.n_hot > 0) FMWR_LAUNCH(ctx, (rm_stats_kernel<T, 2>), grid, 256, 0, a);
      else FMWR_LAUNCH(ctx, (rm_stats_kernel<T, 0>), grid, 256, 0, a);
    }
    if (ctx->nccl_comm && ctx->world > 1) comm_allreduce_sum(ctx, a.AB, 2 * (size_t)a.ncols, sizeof(T) == 8);
    { PeerArgs nopeer; memset(&nopeer, 0, sizeof nopeer); FMWR_LAUNCH(ctx, rm_solve_kernel<T>, ceil_div(a.ncols, 256), 256, 0, a, nopeer, 0); }
    if (a.pe > a.pb) {
      const int grid = (int)std::min<int64_t>(grid_stream, ceil_div64(a.pe - a.pb, 256));
      FMWR_LAUNCH(ctx, rm_apply_kernel<T>, grid, 256, 0, a);
    }
  }
}


// ---- dense (field-structured) fused passes ------------------------------------------------------------------------
// When every row holds exactly one non-zero of every phase (one-hot fields: user/item/context, Criteo's 39 fields) the
// phase's entries are stored [phase][row] with the row implicit, and consecutive coordinate steps are FUSED per row:
//   fused(t) = apply(step t-1) ; stats(step t)
// e[r] (and q_f[r] when both steps belong to the same factor) is read once and written once per step instead of being
// read by stats, then read and written again by apply: 32 instead of 48 bytes per row and step, all of it 128-bit
// coalesced streams (4 rows per thread).
template <class T>
struct StepScratch { T* th; T* AB; T* delta; typename Vec2<T>::type* thd; };

template <class T>
struct FusedArgs {
  int64_t n;
  T* e;
  int has_prev; const uint32_t* pcol; const float* pval; const typename Vec2<T>::type* pthd; T* pq;
  int has_cur; const uint32_t* ccol; const float* cval; const T* cth; T* cAB; T* cq;
  uint32_t p_ncols, c_ncols; int n_rep;
  int cur_sorted;      // the rows are sorted by the current field: equal features sit in consecutive rows
};

constexpr int FUSED_THREADS = 512;
constexpr int FUSED_BLOCKS = 3;             // resident CTAs per SM
constexpr int FUSED_MAX_REP = 64;           // replicas of the per-feature (A, B) table
constexpr size_t FUSED_AB_BYTES = 8u << 20; // ... as many as fit this budget (L2-resident)

// Statistics go to global memory with ONE native 8-byte vector reduction per run (red.global.add.v2.f32).  Shared-memory
// float atomics are compare-and-swap loops on this architecture (ATOMS.CAST.SPIN) and cost more than the whole streaming
// pass; the global reduction unit is spread over n_rep copies of the table (chosen so that they stay L2-resident), which
// keeps same-address serialisation negligible even for a 2048-feature field.  A thread owns VEC consecutive rows and first
// combines the rows that share a feature -- with the rows sorted by the widest field that is one reduction per thread.
// ONES: every value of the data is 1.0 (one-hot fields): the value streams are not read at all.
// apply(step t-1) and the per-row statistics of step t for the VEC rows starting at `base`
// (reference :251-253 / :338-349 for the apply, :225-230 / :313-321 for the statistics)
template <class T, int VEC, bool ONES>
__device__ __forceinline__ void fused_rows(const FusedArgs<T>& a, int64_t base, bool same_q, uint32_t (&cc)[VEC], T (&sa)[VEC], T (&sb)[VEC])
{
  typedef typename Vec2<T>::type V2;
  typedef typename Vec<T>::type V16;
  // (staging these lookup tables in shared memory was measured and does not pay: the pass is bound by the reductions)
  const V2* __restrict__ ptab = a.pthd;
  const T* __restrict__ ctab = a.cth;
  T ev[VEC], qv[VEC];
  uint32_t pc[VEC];
  float px[VEC], cx[VEC];
#pragma unroll
  for (int u = 0; u < VEC; ++u) { px[u] = 1.f; cx[u] = 1.f; pc[u] = 0u; cc[u] = 0u; }
  if (VEC == 4) {
    *reinterpret_cast<V16*>(ev) = *reinterpret_cast<const V16*>(a.e + base);
    if (sizeof(T) == 8) *reinterpret_cast<V16*>(ev + 2) = *reinterpret_cast<const V16*>(a.e + base + 2);
    if (a.has_prev) {
      *reinterpret_cast<uint4*>(pc) = *reinterpret_cast<const uint4*>(a.pcol + base);
      if (!ONES) *reinterpret_cast<float4*>(px) = *reinterpret_cast<const float4*>(a.pval + base);
    }
    if (a.has_cur) {
      *reinterpret_cast<uint4*>(cc) = *reinterpret_cast<const uint4*>(a.ccol + base);
      if (!ONES) *reinterpret_cast<float4*>(cx) = *reinterpret_cast<const float4*>(a.cval + base);
    }
  } else {
    ev[0] = a.e[base];
    if (a.has_prev) { pc[0] = a.pcol[base]; if (!ONES) px[0] = a.pval[base]; }
    if (a.has_cur) { cc[0] = a.ccol[base]; if (!ONES) cx[0] = a.cval[base]; }
  }
  if (a.has_prev) {
    if (a.pq != nullptr) {
      if (VEC == 4 && sizeof(T) == 4) *reinterpret_cast<V16*>(qv) = *reinterpret_cast<const V16*>(a.pq + base);
      else {
#pragma unroll
        for (int u = 0; u < VEC; ++u) qv[u] = a.pq[base + u];
      }
#pragma unroll
      for (int u = 0; u < VEC; ++u) {
        const V2 td = ptab[pc[u]];
        const T d = td.y;
        const T h = T(px[u]) * qv[u] - T(px[u] * px[u]) * td.x;
        qv[u] -= T(px[u]) * d;
        ev[u] -= h * d;
      }
      if (VEC == 4 && sizeof(T) == 4) *reinterpret_cast<V16*>(a.pq + base) = *reinterpret_cast<const V16*>(qv);
      else {
#pragma unroll
        for (int u = 0; u < VEC; ++u) a.pq[base + u] = qv[u];
      }
    } else {
#pragma unroll
      for (int u = 0; u < VEC; ++u) ev[u] -= T(px[u]) * ptab[pc[u]].y;
    }
    if (VEC == 4 && sizeof(T) == 4) *reinterpret_cast<V16*>(a.e + base) = *reinterpret_cast<const V16*>(ev);
    else {
#pragma unroll
      for (int u = 0; u < VEC; ++u) a.e[base + u] = ev[u];
    }
  }
#pragma unroll
  for (int u = 0; u < VEC; ++u) { sa[u] = T(0); sb[u] = T(0); }
  if (a.has_cur) {
    if (a.cq != nullptr && !same_q) {
      if (VEC == 4 && sizeof(T) == 4) *reinterpret_cast<V16*>(qv) = *reinterpret_cast<const V16*>(a.cq + base);
      else {
#pragma unroll
        for (int u = 0; u < VEC; ++u) qv[u] = a.cq[base + u];
      }
    }
#pragma unroll
    for (int u = 0; u < VEC; ++u) {
      const T old = ctab[cc[u]];
      if (a.cq == nullptr) {
        const T x = T(cx[u]);
        sa[u] = x * x;
        sb[u] = ev[u] * x - old * x * x;
      } else {
        const T h = T(cx[u]) * qv[u] - T(cx[u] * cx[u]) * old;
        sa[u] = h * h;
        sb[u] = h * ev[u];
      }
    }
  }
}

template <class T, int VEC, bool ONES>
__global__ void __launch_bounds__(FUSED_THREADS, FUSED_BLOCKS) fused_kernel(FusedArgs<T> a)
{
  const bool same_q = a.has_prev && a.has_cur && a.pq != nullptr && a.pq == a.cq;
  T* AB = a.cAB + (a.has_cur ? 2 * (size_t)(blockIdx.x % (unsigned)a.n_rep) * a.c_ncols : 0);
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * VEC;
  // the loop condition is warp-uniform (first lane's row), so every lane reaches the shuffles of the sorted-field path
  for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC; base - (int64_t)lane * VEC < a.n; base += stride) {
    const bool valid = base < a.n;
    uint32_t cc[VEC];
    T sa[VEC], sb[VEC];
    if (valid) fused_rows<T, VEC, ONES>(a, base, same_q, cc, sa, sb);
    if (!a.has_cur) continue;
    T ra = T(0), rb = T(0);
    uint32_t rc = valid ? cc[0] : 0u;
    bool single = valid;
    if (valid) {
#pragma unroll
      for (int u = 0; u < VEC; ++u) {
        if (u > 0 && cc[u] != rc) { atomic_add2(AB, rc, ra, rb); rc = cc[u]; ra = T(0); rb = T(0); single = false; }
        ra += sa[u]; rb += sb[u];
      }
    }
    if (a.cur_sorted) {
      // Rows are sorted by this field, so the lanes whose rows all carry the previous lane's feature continue its run.
      // A segmented shuffle reduction leaves each run's total in its first lane: ~2 reductions per warp instead of 32.
      // (A thread that saw a feature change has already emitted its earlier runs and starts a new segment with its last.)
      const uint32_t prev_rc = __shfl_up_sync(0xffffffffu, rc, 1);
      const bool head = lane == 0 || !valid || !single || prev_rc != rc;
      const unsigned heads = __ballot_sync(0xffffffffu, head);
      const int seg = __popc(heads & (0xffffffffu >> (31 - lane)));          // heads at or below this lane
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const T ta = __shfl_down_sync(0xffffffffu, ra, o);
        const T tb = __shfl_down_sync(0xffffffffu, rb, o);
        const int ts = __shfl_down_sync(0xffffffffu, seg, o);
        if (lane + o < 32 && ts == seg) { ra += ta; rb += tb; }
      }
      if (valid && head) atomic_add2(AB, rc, ra, rb);
    } else if (valid) {
      atomic_add2(AB, rc, ra, rb);
    }
  }
}

struct DenseLayout {
  bool ok = false;
  DBuf<uint32_t> col;    // [n_phases][n] phase-local feature id
  DBuf<float> val;       // [n_phases][n]
  // optional row permutation: rows sorted by the feature of the widest phase (so that phase needs ~1 atomic per
  // run instead of per row).  e, q and the labels then live in permuted row order; parameters are unaffected.
  bool permuted = false;
  int sorted_phase = -1;
  bool all_ones = false;  // every stored value is 1.0f: the fused passes skip the value streams
  DBuf<uint32_t> pcol;   // [n][np] CSR columns of the permuted rows (global ids) for the forward pass
  DBuf<float> pval;      // [n][np]
  DBuf<float> py;        // [n] labels of the permuted rows
  DBuf<uint32_t> perm;   // [n] original row of permuted row i (the posterior mean un-permutes its row sums with it)
};

__global__ void dense_check_kernel(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, int64_t n, int np,
                                   const uint32_t* __restrict__ pbeg, int* __restrict__ bad)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  if (rowptr[r] != (uint32_t)(r * np) || rowptr[r + 1] != (uint32_t)((r + 1) * np)) { *bad = 1; return; }
  for (int j = 0; j < np; ++j) {
    const uint32_t c = col[r * np + j];
    if (c < pbeg[j] || c >= pbeg[j + 1]) { *bad = 1; return; }
  }
}

__global__ void dense_build_kernel(const uint32_t* __restrict__ col, const float* __restrict__ val, int64_t n, int np,
                                   const uint32_t* __restrict__ pbeg, const uint32_t* __restrict__ perm,
                                   uint32_t* __restrict__ ocol, float* __restrict__ oval)
{
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // output-major: t = j * n + i
  if (t >= n * np) return;
  const int64_t j = t / n, i = t - j * n;
  const int64_t r = perm ? (int64_t)perm[i] : i;
  ocol[t] = col[r * np + j] - pbeg[j];
  oval[t] = val[r * np + j];
}

__global__ void dense_not_one_kernel(const float* __restrict__ val, int64_t m, int* __restrict__ flag)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m && val[i] != 1.0f) *flag = 1;
}

__global__ void dense_phase_key_kernel(const uint32_t* __restrict__ col, int64_t n, int np, int j, uint32_t* __restrict__ key)
{
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n) key[r] = col[r * np + j];
}

__global__ void dense_permute_rows_kernel(const uint32_t* __restrict__ col, const float* __restrict__ val, const float* __restrict__ y,
                                          int64_t n, int np, const uint32_t* __restrict__ perm, uint32_t* __restrict__ pcol,
                                          float* __restrict__ pval, float* __restrict__ py)
{
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // t = i * np + j
  if (t >= n * np) return;
  const int64_t i = t / np, j = t - i * np;
  const int64_t r = perm[i];
  pcol[t] = col[r * np + j];
  pval[t] = val[r * np + j];
  if (j == 0) py[i] = y[r];
}

static void build_dense(fmwr_data* d, const std::vector<uint32_t>& pbeg_host, DenseLayout& dl, bool allow_perm)
{
  fmwr_ctx* ctx = d->ctx;
  const int np = (int)pbeg_host.size() - 1;
  const int64_t n = d->n;
  dl.ok = false;
  if (np <= 0 || n <= 0 || d->nnz != n * np) return;
  DBuf<uint32_t> pbeg;
  DBuf<int> bad;
  pbeg.alloc(np + 1); bad.alloc(1);
  bad.zero(ctx->stream);
  FMWR_CUDA(cudaMemcpyAsync(pbeg.p, pbeg_host.data(), 4 * (np + 1), cudaMemcpyHostToDevice, ctx->stream));
  FMWR_LAUNCH(ctx, dense_check_kernel, ceil_div(n, 256), 256, 0, d->rowptr.p, d->col.p, n, np, pbeg.p, bad.p);
  int hbad = 1;
  FMWR_CUDA(cudaMemcpyAsync(&hbad, bad.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  if (hbad) return;
  // widest phase: if it does not fit the shared-memory table, sort the rows by its feature
  int jstar = 0;
  for (int j = 1; j < np; ++j) if (pbeg_host[j + 1] - pbeg_host[j] > pbeg_host[jstar + 1] - pbeg_host[jstar]) jstar = j;
  DBuf<uint32_t>& perm = dl.perm;
  dl.permuted = false; dl.sorted_phase = -1;
  if (allow_perm && pbeg_host[jstar + 1] - pbeg_host[jstar] > (uint32_t)RM_SMEM_COLS && d->has_labels) {
    DBuf<uint32_t> key_in, key_out, idx_in;
    key_in.alloc(n); key_out.alloc(n); idx_in.alloc(n); perm.alloc(n);
    FMWR_LAUNCH(ctx, dense_phase_key_kernel, ceil_div(n, 256), 256, 0, d->col.p, n, np, jstar, key_in.p);
    launch_iota(ctx, idx_in.p, n);
    int bits = 1;
    while (bits < 32 && (1ull << bits) < (uint64_t)pbeg_host[np]) ++bits;
    sort_pairs_u32(ctx, key_in.p, key_out.p, idx_in.p, perm.p, n, bits);
    dl.pcol.alloc((size_t)n * np); dl.pval.alloc((size_t)n * np); dl.py.alloc(n);
    FMWR_LAUNCH(ctx, dense_permute_rows_kernel, ceil_div(n * np, 256), 256, 0, d->col.p, d->val.p, d->y.p, n, np, perm.p, dl.pcol.p,
                dl.pval.p, dl.py.p);
    dl.permuted = true; dl.sorted_phase = jstar;
  }
  dl.col.alloc((size_t)n * np); dl.val.alloc((size_t)n * np);
  FMWR_LAUNCH(ctx, dense_build_kernel, ceil_div(n * np, 256), 256, 0, d->col.p, d->val.p, n, np, pbeg.p, dl.permuted ? perm.p : nullptr,
              dl.col.p, dl.val.p);
  {
    DBuf<int> flag;
    flag.alloc(1);
    flag.zero(ctx->stream);
    FMWR_LAUNCH(ctx, dense_not_one_kernel, ceil_div(n * np, 256), 256, 0, d->val.p, n * np, flag.p);
    int hf = 1;
    FMWR_CUDA(cudaMemcpyAsync(&hf, flag.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    dl.all_ones = hf == 0;
  }
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  dl.ok = true;
}

template <class T>
static int fused_replicas(uint32_t ncols, int grid)
{
  const size_t per = 2 * sizeof(T) * (size_t)std::max<uint32_t>(ncols, 1);
  return (int)std::max<size_t>(1, std::min<size_t>({(size_t)FUSED_MAX_REP, (size_t)grid, FUSED_AB_BYTES / per}));
}
template <class T>
static size_t fused_ab_elems(uint32_t max_cols) { return std::max<size_t>(2 * (size_t)max_cols, FUSED_AB_BYTES / sizeof(T)); }

// row-sharded multi-GPU: sum the table's replicas into replica 0 (and clear the others) so that ONE all-reduce of
// 2 * ncols values per coordinate step carries this rank's statistics
template <class T>
__global__ void ab_collapse_kernel(T* __restrict__ AB, uint32_t ncols, int n_rep)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;        // index into the interleaved [2 * ncols] table
  if (i >= 2 * ncols) return;
  T s = AB[i];
  for (int r = 1; r < n_rep; ++r) { s += AB[(size_t)r * 2 * ncols + i]; AB[(size_t)r * 2 * ncols + i] = T(0); }
  AB[i] = s;
}

// Row-sharded multi-GPU with peer windows: the all-reduce of a coordinate step's statistics is done by our own kernels.
// Every rank sums its replicas and stores the [2 * ncols] table into slot `rank` of EVERY rank's window (NVLink stores),
// then publishes an epoch flag; the solve kernel of the step waits for all flags and sums the `world` slots in rank order
// -- it simply sees them as `world` replicas -- so all ranks compute bit-identical parameters.  No NCCL call, ~10 us of
// latency per step instead of an all-reduce's 40-50.
template <class T>
__global__ void __launch_bounds__(256) ab_push_kernel(const T* __restrict__ AB, uint32_t ncols, int n_rep, PeerArgs pa, size_t buf_off,
                                                      size_t slot_bytes)
{
  const uint32_t n2 = 2 * ncols;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += gridDim.x * blockDim.x) {
    T s = AB[i];
    for (int r = 1; r < n_rep; ++r) s += AB[(size_t)r * n2 + i];
#pragma unroll
    for (int h = 0; h < 8; ++h)
      if (h < pa.world) reinterpret_cast<T*>(pa.base[h] + buf_off + (size_t)pa.rank * slot_bytes)[i] = s;
  }
  peer_signal(pa, PEER_FLAG1, PEER_EPOCH1, PEER_COUNT1);
}

// sum of a host double over the ranks (identical bits on every rank afterwards)
static double allreduce_scalar(fmwr_ctx* ctx, double x)
{
  if (!(ctx->nccl_comm && ctx->world > 1)) return x;
  ctx->red_scratch.ensure(1024);
  FMWR_CUDA(cudaMemcpyAsync(ctx->red_scratch.p, &x, 8, cudaMemcpyHostToDevice, ctx->stream));
  comm_allreduce_sum(ctx, ctx->red_scratch.p, 1, true);
  double r = 0;
  FMWR_CUDA(cudaMemcpyAsync(&r, ctx->red_scratch.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  return r;
}

// one coordinate step of a fused sequence
template <class T>
struct Step { int phase; T* q; int f; T* theta; int64_t stride; double lambda, mu; int w_sd_is_var; long long normal_base; };

template <class T>
static void run_steps_dense(fmwr_ctx* ctx, const std::vector<uint32_t>& pbeg, const RowMajor& rm, const DenseLayout& dl, int64_t n,
                            T* e, const std::vector<Step<T>>& steps, StepScratch<T> sc[2], double alpha, int do_sample,
                            const double* normals, long long n_normals, uint64_t seed)
{
  const int vec = (n % 4 == 0) ? 4 : 1;
  const int grid = (int)std::min<int64_t>((int64_t)ctx->sm_count * FUSED_BLOCKS, ceil_div64(ceil_div64(n, vec), FUSED_THREADS));
  const int T_ = (int)steps.size();
  // peer windows (row-sharded multi-GPU): slots of 2 * max_cols values per rank, two buffers
  PeerArgs pa;
  memset(&pa, 0, sizeof pa);
  uint32_t max_cols = 1;
  for (size_t j = 0; j + 1 < pbeg.size(); ++j) max_cols = std::max(max_cols, pbeg[j + 1] - pbeg[j]);
  const size_t slot_bytes = ((size_t)2 * max_cols * sizeof(T) + 255) & ~(size_t)255;
  const bool use_peer = ctx->nccl_comm && ctx->world > 1 && ctx->peer.ready &&
                        PEER_CTL_BYTES + 2 * (size_t)ctx->world * slot_bytes <= ctx->peer.bytes;
  if (use_peer) {
    pa.rank = ctx->rank; pa.world = ctx->world;
    for (int r = 0; r < ctx->world; ++r) pa.base[r] = (char*)ctx->peer.base[r];
  }
  auto step_args = [&](int t) {
    RmArgs<T> ra;                      // extract / solve arguments of step t
    memset(&ra, 0, sizeof ra);
    const Step<T>& cs = steps[t];
    const uint32_t cb = pbeg[cs.phase], ncols = pbeg[cs.phase + 1] - cb;
    ra.cb = cb; ra.ncols = ncols; ra.q = cs.q; ra.n = n; ra.f = cs.f; ra.theta = cs.theta; ra.theta_stride = cs.stride;
    ra.th = sc[t & 1].th; ra.AB = sc[t & 1].AB; ra.delta = sc[t & 1].delta; ra.thd = sc[t & 1].thd;
    ra.n_rep = fused_replicas<T>(ncols, grid);
    ra.alpha = alpha; ra.lambda = cs.lambda; ra.mu = cs.mu; ra.do_sample = do_sample; ra.w_sd_is_var = cs.w_sd_is_var;
    ra.normals = normals; ra.n_normals = n_normals; ra.normal_base = cs.normal_base; ra.seed = seed;
    return ra;
  };
  RmArgs<T> ra, rnext;
  memset(&ra, 0, sizeof ra);
  if (T_ > 0) {
    rnext = step_args(0);
    FMWR_LAUNCH(ctx, rm_extract_kernel<T>, ceil_div(rnext.ncols, 256), 256, 0, rnext);
  }
  for (int t = 0; t <= T_; ++t) {
    FusedArgs<T> fa;
    memset(&fa, 0, sizeof fa);
    fa.n = n; fa.e = e; fa.n_rep = 1;
    if (t > 0) {
      const Step<T>& ps = steps[t - 1];
      fa.has_prev = 1;
      fa.pcol = dl.col.p + (size_t)ps.phase * n; fa.pval = dl.val.p + (size_t)ps.phase * n;
      fa.pthd = sc[(t - 1) & 1].thd; fa.p_ncols = pbeg[ps.phase + 1] - pbeg[ps.phase];
      fa.pq = ps.q ? ps.q + (size_t)ps.f * n : nullptr;
    }
    if (t < T_) {
      ra = rnext;                      // extracted by the previous iteration's solve+extract launch
      const Step<T>& cs = steps[t];
      fa.has_cur = 1;
      fa.ccol = dl.col.p + (size_t)cs.phase * n; fa.cval = dl.val.p + (size_t)cs.phase * n;
      fa.cth = ra.th; fa.cAB = ra.AB; fa.cq = cs.q ? cs.q + (size_t)cs.f * n : nullptr;
      fa.c_ncols = ra.ncols; fa.n_rep = ra.n_rep;
      fa.cur_sorted = (dl.permuted && dl.sorted_phase == cs.phase && getenv("FMWR_ALS_NO_WARPSEG") == nullptr) ? 1 : 0;
    }
    if (vec == 4) {
      if (dl.all_ones) FMWR_LAUNCH(ctx, (fused_kernel<T, 4, true>), grid, FUSED_THREADS, 0, fa);
      else FMWR_LAUNCH(ctx, (fused_kernel<T, 4, false>), grid, FUSED_THREADS, 0, fa);
    } else {
      if (dl.all_ones) FMWR_LAUNCH(ctx, (fused_kernel<T, 1, true>), grid, FUSED_THREADS, 0, fa);
      else FMWR_LAUNCH(ctx, (fused_kernel<T, 1, false>), grid, FUSED_THREADS, 0, fa);
    }
    RmArgs<T> rs = ra;                 // what solve(t) reads
    int peer_wait_flag = 0;
    if (t < T_ && ctx->nccl_comm && ctx->world > 1) {
      // rows are sharded over the ranks: every rank holds partial (A, B); one exchange per coordinate step (SURVEY 8e)
      if (use_peer) {
        // double-buffered by the parity of a step counter that runs across calls (every rank executes the same sequence):
        // between two pushes into one buffer lies a step whose solve waited for every peer, so nobody still reads it
        const size_t buf_off = PEER_CTL_BYTES + (size_t)(ctx->peer.als_step++ & 1u) * ctx->world * slot_bytes;
        const int pgrid = (int)std::min<int64_t>(ceil_div(2 * (int64_t)ra.ncols, 256), ctx->sm_count * 2);
        FMWR_LAUNCH(ctx, ab_push_kernel<T>, pgrid, 256, 0, ra.AB, ra.ncols, ra.n_rep, pa, buf_off, slot_bytes);
        rs.AB = reinterpret_cast<T*>(pa.base[pa.rank] + buf_off);
        rs.n_rep = ctx->world;         // the ranks' tables, slot_bytes apart ...
        rs.rep_stride = slot_bytes / (2 * sizeof(T));    // ... in units of (A, B) pairs
        peer_wait_flag = 1;
      } else {
        if (ra.n_rep > 1) FMWR_LAUNCH(ctx, ab_collapse_kernel<T>, ceil_div(2 * (int64_t)ra.ncols, 256), 256, 0, ra.AB, ra.ncols, ra.n_rep);
        comm_allreduce_sum(ctx, ra.AB, 2 * (size_t)ra.ncols, sizeof(T) == 8);
      }
    }
    if (t < T_) {
      if (t + 1 < T_) {
        // solve(t) and extract(t+1) share a launch: step t+1 is another (phase, factor), i.e. other features, and its
        // scratch (parity (t+1)&1) was last read by the fused pass that has just finished
        rnext = step_args(t + 1);
        FMWR_LAUNCH(ctx, rm_solve_extract_kernel<T>, ceil_div(std::max(ra.ncols, rnext.ncols), SE_COLS), SE_COLS * SE_SLICES, 0, rs, rnext, pa,
                    peer_wait_flag);
      } else FMWR_LAUNCH(ctx, rm_solve_kernel<T>, ceil_div(ra.ncols, 256), 256, 0, rs, pa, peer_wait_flag);
    }
  }
}

// ---- driver ----------------------------------------------------------------------------------------------
struct PhaseInfo {
  std::vector<uint32_t> begin;                 // [n_phases + 1]
  std::vector<std::vector<uint32_t>> long_cols;
  DBuf<uint32_t> long_dev;                     // concatenated
  std::vector<uint32_t> colptr_host;
  std::vector<size_t> long_off;
};

static void build_phase_info(fmwr_data* d, PhaseInfo& ph)
{
  fmwr_ctx* ctx = d->ctx;
  phases_build(d);
  ph.begin = d->phase_begin;
  const int np = (int)ph.begin.size() - 1;
  std::vector<uint32_t> cp(d->p + 1);
  FMWR_CUDA(cudaMemcpyAsync(cp.data(), d->colptr.p, 4 * (d->p + 1), cudaMemcpyDeviceToHost, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  ph.colptr_host = cp;
  std::vector<uint32_t> all;
  ph.long_off.assign(np + 1, 0);
  for (int i = 0; i < np; ++i) {
    ph.long_off[i] = all.size();
    for (uint32_t c = ph.begin[i]; c < ph.begin[i + 1]; ++c)
      if (cp[c + 1] - cp[c] >= (uint32_t)ALS_LONG) all.push_back(c);
  }
  ph.long_off[np] = all.size();
  ph.long_dev.alloc(all.size());
  if (!all.empty()) FMWR_CUDA(cudaMemcpyAsync(ph.long_dev.p, all.data(), 4 * all.size(), cudaMemcpyHostToDevice, ctx->stream));
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
}

template <class T>
static void run_phases(fmwr_ctx* ctx, const PhaseInfo& ph, CoordArgs<T> a)
{
  const int np = (int)ph.begin.size() - 1;
  for (int i = 0; i < np; ++i) {
    a.c_begin = ph.begin[i]; a.c_end = ph.begin[i + 1];
    const uint32_t nc = a.c_end - a.c_begin;
    if (nc == 0) continue;
    FMWR_LAUNCH(ctx, coord_warp_kernel<T>, ceil_div(nc, 8), 256, 0, a);
    const int nl = (int)(ph.long_off[i + 1] - ph.long_off[i]);
    if (nl > 0) {
      a.long_cols = ph.long_dev.p + ph.long_off[i]; a.n_long = nl;
      FMWR_LAUNCH(ctx, coord_block_kernel<T>, nl, 512, 0, a);
    }
  }
}

struct HostStreams {
  const double* normals; long long n_normals, i_normal;
  const double* gammas; long long n_gammas, i_gamma;
  std::mt19937_64 rng;
  bool injected;
  double normal(double mean, double sd)
  {
    double z;
    if (injected) { z = (normals && i_normal < n_normals) ? normals[i_normal] : 0.0; }
    else { std::normal_distribution<double> nd(0.0, 1.0); z = nd(rng); }
    i_normal++;
    return mean + sd * z;
  }
  double gamma(double shape, double scale)
  {
    double g;
    if (injected) { g = (gammas && i_gamma < n_gammas) ? gammas[i_gamma] : 1.0; }
    else { std::gamma_distribution<double> gd(shape, 1.0); g = gd(rng); }
    i_gamma++;
    return scale * g;
  }
};

static inline bool hbad(double x) { return std::isnan(x) || std::isinf(x); }

template <class T>
static void train_als_t(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Posterior* post,
                        const Holdout* holdout)
{
  const int64_t n = d->n, p = d->p;
  const int k = m->k, kp = m->kp;
  const bool mcmc = s->solver == FMWR_MCMC;
  const bool do_sample = mcmc, do_multilevel = mcmc;                     // reference :567-587
  const bool cls = m->cfg.task == FMWR_CLASSIFICATION;
  const bool enable_v = s->enable_v && k > 0;
  FMWR_REQUIRE(n < (1ll << 31) && p < (1ll << 31), FMWR_ERR_UNSUPPORTED, "dimension too large");

  // Row-sharded multi-GPU (communicator initialised): the data handle is this rank's ROWS, the model is replicated.
  // Every rank runs the same sweep; per-feature statistics and the two residual sums are all-reduced, so all ranks
  // derive bit-identical parameters (and, for MCMC, identical draws: same seeds, same reduced inputs).
  const bool multi = ctx->nccl_comm != nullptr && ctx->world > 1;
  double n_glob = (double)n;
  int64_t row_off = 0;
  if (multi) {
    FMWR_REQUIRE(s->step_size <= 0, FMWR_ERR_UNSUPPORTED, "the tracker is not available on row-sharded data (score the shards separately)");
    FMWR_REQUIRE(!s->rands, FMWR_ERR_UNSUPPORTED, "an injected rand() stream is consumed in global row order: single GPU only");
    ctx->red_scratch.ensure(1024);
    std::vector<double> cnt(ctx->world, 0.0);
    cnt[ctx->rank] = (double)n;
    FMWR_CUDA(cudaMemcpyAsync(ctx->red_scratch.p, cnt.data(), 8 * ctx->world, cudaMemcpyHostToDevice, ctx->stream));
    comm_allreduce_sum(ctx, ctx->red_scratch.p, ctx->world, true);
    FMWR_CUDA(cudaMemcpyAsync(cnt.data(), ctx->red_scratch.p, 8 * ctx->world, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    n_glob = 0;
    for (int r = 0; r < ctx->world; ++r) { if (r < ctx->rank) row_off += (int64_t)cnt[r]; n_glob += cnt[r]; }
  }

  transpose_build(d);                                                    // src/FM.cpp:148-152
  struct AlsCache { PhaseInfo ph; RowMajor rm; DenseLayout dl; bool rm_tried = false; };
  if (d->als_cache && s->rands && static_cast<AlsCache*>(d->als_cache.get())->dl.permuted) d->als_cache.reset();
  if (!d->als_cache) {
    auto c = std::make_shared<AlsCache>();
    build_phase_info(d, c->ph);
    d->als_cache = c;
  }
  AlsCache& cache = *static_cast<AlsCache*>(d->als_cache.get());
  PhaseInfo& ph = cache.ph;

  // streaming (row-major) coordinate passes when the data decomposes into few phases (field-structured data);
  // otherwise the column-parallel kernels
  RowMajor& rm = cache.rm;
  const int n_phases = (int)ph.begin.size() - 1;
  const bool use_rm = n_phases <= 256 && d->nnz > 0 && getenv("FMWR_ALS_COLUMN") == nullptr;
  FMWR_REQUIRE(!multi || use_rm, FMWR_ERR_UNSUPPORTED, "row-sharded ALS/MCMC needs phase-decomposable (field-structured) data");
  DBuf<T> rm_th, rm_AB, rm_delta, rm_th2, rm_AB2, rm_delta2, rm_thd, rm_thd2;
  DenseLayout& dl = cache.dl;
  if (use_rm) {
    if (!cache.rm_tried) {
      build_row_major(d, ph.begin, ph.colptr_host, rm);
      // (an injected rand() stream is consumed in ORIGINAL row order, so such validation runs keep the rows unpermuted)
      if (getenv("FMWR_ALS_NO_DENSE") == nullptr) build_dense(d, ph.begin, dl, s->rands == nullptr && getenv("FMWR_ALS_NO_PERM") == nullptr);
      if (dl.ok) { rm.row.release(); rm.col.release(); rm.val.release(); }     // the dense copy supersedes the row-major one
      cache.rm_tried = true;
    }
    rm_th.alloc(rm.max_cols); rm_AB.alloc(dl.ok ? fused_ab_elems<T>(rm.max_cols) : 2 * (size_t)rm.max_cols); rm_delta.alloc(rm.max_cols);
    if (dl.ok) { rm_th2.alloc(rm.max_cols); rm_AB2.alloc(fused_ab_elems<T>(rm.max_cols)); rm_delta2.alloc(rm.max_cols); rm_thd.alloc(2 * (size_t)rm.max_cols); rm_thd2.alloc(2 * (size_t)rm.max_cols); }
  }
  typedef typename Vec2<T>::type V2T;
  StepScratch<T> scr[2] = {{rm_th.p, rm_AB.p, rm_delta.p, (V2T*)rm_thd.p}, {rm_th2.p, rm_AB2.p, rm_delta2.p, (V2T*)rm_thd2.p}};
  auto rm_args = [&](T* e_p, T* q_p, int f, T* theta, int64_t stride, double alpha_, double lambda_, double mu_, int sample, int w_sd_var,
                     const double* normals_p, long long n_normals_, long long base, uint64_t seed_) {
    RmArgs<T> a;
    memset(&a, 0, sizeof a);
    a.row = rm.row.p; a.col = rm.col.p; a.val = rm.val.p; a.hot = rm.hot.p;
    a.e = e_p; a.q = q_p; a.n = n; a.f = f; a.theta = theta; a.theta_stride = stride;
    a.th = rm_th.p; a.AB = rm_AB.p; a.delta = rm_delta.p;
    a.alpha = alpha_; a.lambda = lambda_; a.mu = mu_; a.do_sample = sample; a.w_sd_is_var = w_sd_var;
    a.normals = normals_p; a.n_normals = n_normals_; a.normal_base = base; a.seed = seed_;
    return a;
  };

  DBuf<T> e, q;
  e.alloc(n);
  if (enable_v) q.alloc((size_t)n * kp);
  DBuf<double> normals_dev;
  DBuf<int32_t> rands_dev;
  DBuf<long long> rand_pos;
  const bool injected = s->normals || s->gammas || s->rands;
  if (s->normals && s->n_normals > 0) {
    normals_dev.alloc(s->n_normals);
    FMWR_CUDA(cudaMemcpyAsync(normals_dev.p, s->normals, 8 * s->n_normals, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (s->rands && s->n_rands > 0) {
    rands_dev.alloc(s->n_rands);
    FMWR_CUDA(cudaMemcpyAsync(rands_dev.p, s->rands, 4 * s->n_rands, cudaMemcpyHostToDevice, ctx->stream));
    rand_pos.alloc(1);
    rand_pos.zero(ctx->stream);
  }
  HostStreams hs{s->normals, (long long)s->n_normals, 0, s->gammas, (long long)s->n_gammas, 0, std::mt19937_64(s->seed ^ 0x5DEECE66Dull), injected};

  // MCMC_ALS_Learner::init (:59-89) -- constants forced regardless of the R-side values (F2)
  const double alpha_0 = 1.0, gamma_0 = 1.0, beta_0 = 1.0, mu_0 = 0.0, w0_mean_0 = 0.0;
  double alpha = 1.0, w_mu = 0.0, w_lambda = 0.0;
  std::vector<double> v_mu(std::max(k, 1), 0.0), v_lambda(std::max(k, 1), 0.0);

  // posterior mean: f64 sums of the predict.FM prediction of every averaged draw (the MCMC link of tracker_score) -- the
  // training rows in the order e has, then each eval set.  Draw t is the model after t sweeps: at sweep t, right after the
  // forward, e holds its raw score; the eval sets get a predict of their own.  None of it feeds back into the chain.
  const int post_link = tracker_link(m->cfg.task, s->solver);
  DBuf<double> post_acc;
  std::vector<int64_t> post_off;           // [n_eval + 2] offsets into post_acc
  if (post) {
    post_off = {0, n};
    for (int i = 0; i < post->n_eval; ++i) post_off.push_back(post_off.back() + post->eval[i]->n);
    post_acc.alloc(post_off.back());
    post_acc.zero(ctx->stream);
  }
  auto post_draw = [&]() {
    if (n > 0)
      FMWR_LAUNCH(ctx, posterior_accum_kernel<T>, ceil_div(n, 256), 256, 0, e.p, n, post_link, s->min_target, s->max_target,
                  ctx->pn_table.p, post_acc.p);
    for (int i = 0; i < post->n_eval; ++i) {
      fmwr_data* ev = post->eval[i];
      if (ev->n == 0) continue;
      forward_launch(ctx, m, ev, FMWR_LINK_NONE, 0.0, 0.0);
      FMWR_LAUNCH(ctx, posterior_accum_kernel<double>, ceil_div(ev->n, 256), 256, 0, ev->pred64.p, ev->n, post_link, s->min_target,
                  s->max_target, ctx->pn_table.p, post_acc.p + post_off[i + 1]);
    }
  };

  T* wp = (T*)m->w.p;
  T* vp = (T*)m->v.p;
  double* scal = (double*)m->scal.p;
  Tracker trk(ctx, m, s, tr, holdout);
  int sweep = 0;
  for (; sweep < s->max_iter; ++sweep) {
    // tracker (:101-124): train metric of the model at the start of the sweep; a stop decided there skips the sweep
    if (trk.due(sweep) && trk.record(sweep, tracker_score(ctx, m, d, s))) break;
    // e <- predict_batch (:100), q[r][f] <- S_f
    const bool perm_rows = use_rm && dl.ok && dl.permuted;     // e, q, labels in permuted row order (see DenseLayout)
    const float* yp = perm_rows ? dl.py.p : d->y.p;
    AlsFwd<T> fw{ctx, m, d, e.p, enable_v ? q.p : nullptr, perm_rows ? dl.pcol.p : d->col.p, perm_rows ? dl.pval.p : d->val.p};
    dispatch_layout<T>(kp, fw);
    if (post && sweep > post->burn_in) post_draw();
    // calculate_error (:520-562)
    if (!cls) {
      FMWR_LAUNCH(ctx, als_error_kernel<T>, ceil_div(n, 256), 256, 0, e.p, yp, n, 0, ctx->dp_table.p, s->seed, (uint64_t)sweep, (uint64_t)row_off);
    } else if (!do_sample) {
      FMWR_LAUNCH(ctx, als_error_kernel<T>, ceil_div(n, 256), 256, 0, e.p, yp, n, 1, ctx->dp_table.p, s->seed, (uint64_t)sweep, (uint64_t)row_off);
    } else if (s->rands) {
      FMWR_LAUNCH(ctx, als_error_stream_kernel<T>, 1, 32, 0, e.p, d->y.p, n, rands_dev.p, (long long)s->n_rands, rand_pos.p);
    } else {
      FMWR_LAUNCH(ctx, als_error_kernel<T>, ceil_div(n, 256), 256, 0, e.p, yp, n, 2, ctx->dp_table.p, s->seed, (uint64_t)sweep, (uint64_t)row_off);
    }
    // update_alpha (:360-380)
    if (!do_multilevel) alpha = alpha_0;
    else {
      const double alpha_n = alpha_0 + n_glob;
      const double gamma_n = gamma_0 + allreduce_scalar(ctx, reduce<T>(ctx, e.p, n, 1, 1, 0.0));
      const double a = hs.gamma(alpha_n / 2.0, 2.0 / gamma_n);
      if (!hbad(a)) alpha = a;
    }
    // update_w0 (:162-188)
    if (m->cfg.keep_w0) {
      const double w0 = model_get_w0(m);
      const double err = allreduce_scalar(ctx, reduce<T>(ctx, e.p, n, 1, 0, 0.0)) - n_glob * w0;
      const double var = 1.0 / (m->cfg.l2_w0 + alpha * n_glob);
      const double mean = -(alpha * err - w0_mean_0 * m->cfg.l2_w0) * var;
      double nw = do_sample ? hs.normal(mean, std::sqrt(var)) : mean;
      if (hbad(nw)) nw = w0;
      FMWR_CUDA(cudaMemcpyAsync(scal, &nw, 8, cudaMemcpyHostToDevice, ctx->stream));
      FMWR_LAUNCH(ctx, als_shift_kernel<T>, ceil_div(n, 256), 256, 0, e.p, n, T(w0 - nw));
      FMWR_CUDA(cudaStreamSynchronize(ctx->stream));      // nw lives on this stack frame
    }
    if (m->cfg.keep_w1) {
      // update_w_lambda (:415-445), update_w_mu (:383-412)
      if (do_multilevel) {
        double g = reduce<T>(ctx, wp, p, 1, 2, w_mu);
        g += beta_0 * (w_mu - mu_0) * (w_mu - mu_0) + gamma_0;
        const double la = alpha_0 + (double)p + 1;
        const double nl = do_sample ? hs.gamma(la / 2.0, 2.0 / g) : la / g;
        if (!hbad(nl)) w_lambda = nl;
        double mm = reduce<T>(ctx, wp, p, 1, 0, 0.0);
        mm = (mm + beta_0 * mu_0) / ((double)p + beta_0);
        const double var = 1.0 / (((double)p + beta_0) * w_lambda);
        const double nm = do_sample ? hs.normal(mm, std::sqrt(var)) : mm;
        if (!hbad(nm)) w_mu = nm;
      } else w_mu = mu_0;
      // update_w (:190-270)
      CoordArgs<T> a;
      memset(&a, 0, sizeof a);
      a.colptr = d->colptr.p; a.crow = d->crow.p; a.cval = d->cval.p;
      a.e = e.p; a.q = nullptr; a.kp = kp; a.f = 0; a.n = n; a.theta = wp; a.theta_stride = 1;
      a.alpha = alpha; a.lambda = w_lambda; a.mu = w_mu; a.do_sample = do_sample;
      a.w_sd_is_var = (s->compat & FMWR_COMPAT_MCMC_W_SD) ? 1 : 0;
      a.normals = injected ? normals_dev.p : nullptr; a.n_normals = s->n_normals; a.normal_base = hs.i_normal; a.seed = s->seed;
      if (use_rm && dl.ok) {
        std::vector<Step<T>> steps;
        for (int j = 0; j < n_phases; ++j) steps.push_back({j, nullptr, 0, wp, 1, w_lambda, w_mu, a.w_sd_is_var, a.normal_base});
        run_steps_dense<T>(ctx, ph.begin, rm, dl, n, e.p, steps, scr, alpha, do_sample, a.normals, a.n_normals, a.seed);
      } else if (use_rm) run_phases_rm<T>(ctx, ph.begin, rm, rm_args(e.p, nullptr, 0, wp, 1, alpha, w_lambda, w_mu, do_sample, a.w_sd_is_var,
                                                               a.normals, a.n_normals, a.normal_base, a.seed));
      else run_phases<T>(ctx, ph, a);
      if (do_sample) hs.i_normal += p;
    }
    if (enable_v) {
      // update_v_lambda (:486-517) for every factor, then update_v_mu (:448-483), then update_v (:272-354)
      if (do_multilevel) {
        // V is not touched between these 2k draws and v_lambda[f] / v_mu[f] only depend on factor f's own sums, so all
        // the sums come from one batched reduction (the draw ORDER -- k lambdas, then k mus -- is the reference's)
        std::vector<double> vsum, vsq, vrow0;
        reduce_v_all<T>(ctx, vp, p, k, kp, v_mu, vsum, vsq, vrow0);
        for (int f = 0; f < k; ++f) {
          double g = vsq[f];
          g += beta_0 * (v_mu[f] - mu_0) * (v_mu[f] - mu_0) + gamma_0;
          const double la = alpha_0 + (double)p + 1;
          const double nl = do_sample ? hs.gamma(la / 2.0, 2.0 / g) : la / g;
          if (!hbad(nl)) v_lambda[f] = nl;
        }
        // F7: the reference sums v(f, attr_group[i]) == v(f, 0), p times (:462).  The p-fold fp64 addition is reproduced
        // exactly, but for all factors at once (k independent chains the CPU can pipeline) -- one factor at a time it
        // was 3 ms of host time per sweep with the GPU idle.
        std::vector<double> vrep(k, 0.0);
        if (s->compat & FMWR_COMPAT_MCMC_VMU_IDX) {
          std::vector<double> v0(k);
          for (int f = 0; f < k; ++f) v0[f] = (double)T(vrow0[f]);
          for (int64_t i = 0; i < p; ++i)
            for (int f = 0; f < k; ++f) vrep[f] += v0[f];
        }
        for (int f = 0; f < k; ++f) {
          double mm = (s->compat & FMWR_COMPAT_MCMC_VMU_IDX) ? vrep[f] : vsum[f];
          mm = (mm + beta_0 * mu_0) / ((double)p + beta_0);
          const double var = 1.0 / (((double)p + beta_0) * v_lambda[f]);
          const double nm = do_sample ? hs.normal(mm, std::sqrt(var)) : mm;
          if (!hbad(nm)) v_mu[f] = nm;
        }
      } else { for (int f = 0; f < k; ++f) v_mu[f] = mu_0; }
      if (use_rm && dl.ok) {
        std::vector<Step<T>> steps;
        for (int f = 0; f < k; ++f) {
          for (int j = 0; j < n_phases; ++j) steps.push_back({j, q.p, f, vp + f, (int64_t)kp, v_lambda[f], v_mu[f], 0, hs.i_normal});
          if (do_sample) hs.i_normal += p;
        }
        run_steps_dense<T>(ctx, ph.begin, rm, dl, n, e.p, steps, scr, alpha, do_sample, injected ? normals_dev.p : nullptr, s->n_normals, s->seed);
      } else
      for (int f = 0; f < k; ++f) {
        CoordArgs<T> a;
        memset(&a, 0, sizeof a);
        a.colptr = d->colptr.p; a.crow = d->crow.p; a.cval = d->cval.p;
        a.e = e.p; a.q = q.p; a.kp = kp; a.f = f; a.n = n; a.theta = vp + f; a.theta_stride = kp;
        a.alpha = alpha; a.lambda = v_lambda[f]; a.mu = v_mu[f]; a.do_sample = do_sample; a.w_sd_is_var = 0;
        a.normals = injected ? normals_dev.p : nullptr; a.n_normals = s->n_normals; a.normal_base = hs.i_normal; a.seed = s->seed;
        if (use_rm) run_phases_rm<T>(ctx, ph.begin, rm, rm_args(e.p, q.p, f, vp + f, kp, alpha, v_lambda[f], v_mu[f], do_sample, 0,
                                                                 a.normals, a.n_normals, a.normal_base, a.seed));
        else run_phases<T>(ctx, ph, a);
        if (do_sample) hs.i_normal += p;
      }
    }
  }
  if (post) {
    // the last draw is the returned model: one more forward (scores only) for the training rows
    const bool perm_rows = use_rm && dl.ok && dl.permuted;
    AlsFwd<T> fw{ctx, m, d, e.p, nullptr, perm_rows ? dl.pcol.p : d->col.p, perm_rows ? dl.pval.p : d->val.p};
    dispatch_layout<T>(kp, fw);
    post_draw();
    const double draws = (double)(s->max_iter - post->burn_in);
    for (int i = -1; i < post->n_eval; ++i) {
      fmwr_data* dd = i < 0 ? d : post->eval[i];
      if (dd->n == 0) continue;
      dd->pred64.ensure(dd->n);
      FMWR_LAUNCH(ctx, posterior_mean_kernel, ceil_div(dd->n, 256), 256, 0, post_acc.p + post_off[i + 1], dd->n, draws,
                  (i < 0 && perm_rows) ? dl.perm.p : nullptr, dd->pred64.p);
      dd->pred_prec = FMWR_F64;
    }
  }
  trk.restore_best();
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ctx->world > 1) peer_check_error(ctx);      // a timed-out exchange means partial (A,B) sums: the replicas have diverged
  trk.write_trace(sweep);
}

// ---- precision policy ------------------------------------------------------------------------------------------------------
// fp32 ALS / MCMC is a throughput mode; two situations make it miss the reference's fp64 results by more than rounding, and in
// both the sweep runs in fp64 on a shadow model instead (the fp32 handle gets the result back):
//   * MCMC classification: the truncated-normal augmentation (reference MCMC_ALS_Learner.h:531-541) takes a data-dependent
//     number of rejection steps -- fp32 noise in e changes which draws are consumed;
//   * a feature with one or two non-zeros: h = x q - x^2 v cancels to rounding noise there and var = 1/(lambda + alpha sum h^2)
//     amplifies it (long-tail one-hot data).
__global__ void col_count_kernel(const uint32_t* __restrict__ col, int64_t nnz, uint32_t* __restrict__ cnt)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) atomicAdd(cnt + col[i], 1u);
}
__global__ void col_count_min_kernel(const uint32_t* __restrict__ cnt, int64_t p, uint32_t* __restrict__ out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t c = 0xffffffffu;
  if (i < p && cnt[i] > 0u) c = cnt[i];
  for (int o = 16; o > 0; o >>= 1) c = min(c, __shfl_xor_sync(0xffffffffu, c, o));
  if ((threadIdx.x & 31) == 0 && c != 0xffffffffu) atomicMin(out, c);
}

static bool has_thin_columns(fmwr_ctx* ctx, fmwr_data* d)
{
  if (d->min_col_nnz < 0) {
    DBuf<uint32_t> cnt, mn;
    cnt.alloc(std::max<int64_t>(d->p, 1)); mn.alloc(1);
    cnt.zero(ctx->stream);
    FMWR_CUDA(cudaMemsetAsync(mn.p, 0xff, 4, ctx->stream));
    if (d->nnz > 0) FMWR_LAUNCH(ctx, col_count_kernel, ceil_div(d->nnz, 256), 256, 0, d->col.p, d->nnz, cnt.p);
    // row shards: a column's count is the sum over the shards (a shard alone sees a fraction of every column and would call
    // almost any data thin); every rank then derives the same answer
    if (ctx->nccl_comm && ctx->world > 1 && d->p > 0) comm_allreduce_sum_u32(ctx, cnt.p, (size_t)d->p);
    if (d->p > 0) FMWR_LAUNCH(ctx, col_count_min_kernel, ceil_div(d->p, 256), 256, 0, cnt.p, d->p, mn.p);
    uint32_t h = 0;
    FMWR_CUDA(cudaMemcpyAsync(&h, mn.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    d->min_col_nnz = h == 0xffffffffu ? (1ll << 40) : (int64_t)h;
  }
  return d->min_col_nnz <= 2;
}

template <class A, class B>
__global__ void repack_rows_kernel(const A* __restrict__ src, int kp_src, B* __restrict__ dst, int kp_dst, int64_t p, int k)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p * kp_dst) return;
  const int f = (int)(i % kp_dst);
  const int64_t j = i / kp_dst;
  dst[i] = f < k ? (B)src[j * kp_src + f] : B(0);
}

int als_effective_precision(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s)
{
  if (m->prec == FMWR_F64) return FMWR_F64;
  if (s->solver == FMWR_MCMC && m->cfg.task == FMWR_CLASSIFICATION) return FMWR_F64;
  return has_thin_columns(ctx, d) ? FMWR_F64 : FMWR_F32;
}

void train_als_mcmc(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Posterior* post,
                    const Holdout* holdout)
{
  if (m->prec == FMWR_F64) { train_als_t<double>(ctx, m, d, s, tr, post, holdout); return; }
  if (als_effective_precision(ctx, m, d, s) == FMWR_F32) { train_als_t<float>(ctx, m, d, s, tr, post, holdout); return; }
  // fp64 shadow of the fp32 handle (a posterior mean averages the shadow's draws; held-out tracking scores the shadow and
  // restores its best copy into the shadow, before the handback below narrows it into the fp32 handle)
  fmwr_model* sh = nullptr;
  FMWR_REQUIRE(fmwr_model_create(ctx, &m->cfg, m->p, FMWR_F64, &sh) == 0, FMWR_ERR_CUDA, fmwr_last_error());
  try {
    const int64_t p = m->p;
    FMWR_CUDA(cudaMemcpyAsync(sh->scal.p, m->scal.p, 8 * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    if (p > 0) {
      FMWR_LAUNCH(ctx, (repack_rows_kernel<float, double>), ceil_div(p, 256), 256, 0, (const float*)m->w.p, 1, (double*)sh->w.p, 1, p, 1);
      FMWR_LAUNCH(ctx, (repack_rows_kernel<float, double>), ceil_div(p * sh->kp, 256), 256, 0, (const float*)m->v.p, m->kp, (double*)sh->v.p, sh->kp, p, m->k);
    }
    train_als_t<double>(ctx, sh, d, s, tr, post, holdout);
    FMWR_CUDA(cudaMemcpyAsync(m->scal.p, sh->scal.p, 8 * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    if (p > 0) {
      FMWR_LAUNCH(ctx, (repack_rows_kernel<double, float>), ceil_div(p, 256), 256, 0, (const double*)sh->w.p, 1, (float*)m->w.p, 1, p, 1);
      FMWR_LAUNCH(ctx, (repack_rows_kernel<double, float>), ceil_div(p * m->kp, 256), 256, 0, (const double*)sh->v.p, sh->kp, (float*)m->v.p, m->kp, p, m->k);
    }
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  } catch (...) { fmwr_model_destroy(sh); throw; }
  fmwr_model_destroy(sh);
}

}  // namespace fmwr
