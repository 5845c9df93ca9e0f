// Warp-per-row FM forward over device CSR.
//
// Replaces Model::predict / Model::predict_batch (reference src/core/Model.h:75-161):
//   y = [k0] w0 + [k1] sum_j w_j x_j + sum_f 1/2 (S_f^2 - Q_f),  S_f = sum_j v_jf x_j,  Q_f = sum_j (v_jf x_j)^2
//
// Layout: V is [p][kp] (feature-major, kp = padded k), so one feature's factors are one or a
// few contiguous 16-byte vectors.  A warp owns a row; it is split into G = 32/LPR groups of LPR
// lanes; a group fetches one V row per step with ONE 128-bit load per lane (k=32 fp32: LPR=8, a
// 128-byte line per group, 4 non-zeros per warp-wide load instruction), U steps are kept in flight.
// Lane l of every group accumulates S and Q for factors [l*VN, l*VN+VN) (+ chunk offsets); groups
// are combined with xor-shuffles at the end of the row.
#pragma once
#include "common.cuh"

namespace fmwr {

// Loads that the compiler must keep in program order (volatile asm): the gather loop issues a whole batch of
// column / value loads, then a whole batch of factor-row loads, and only then consumes them.  Left to itself the
// compiler sinks every load next to its first use, which serialises the batch into one dependent round per entry.
__device__ __forceinline__ uint32_t ld_nc_u32(const uint32_t* p) { uint32_t r; asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }
__device__ __forceinline__ float ld_nc_f32(const float* p) { float r; asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p)); return r; }
__device__ __forceinline__ float4 ld_nc_v16(const float4* p)
{
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ double2 ld_nc_v16(const double2* p)
{
  double2 r;
  asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}

// ---- team forward ------------------------------------------------------------------------------------------
// A TEAM of lanes owns a row: the whole warp (TEAM = 32; long rows) or one LPR-lane group (TEAM = LPR; rows with a
// handful of non-zeros, 32/LPR rows per warp).  The team is NG = TEAM/LPR sub-groups; sub-group sg fetches entries
// sg, sg + NG, ... of the row, U factor rows in flight.  These kernels are instruction-issue bound, so the loop is
// written for instruction count: immediate-offset loads off a running pointer, an unpredicated path for full
// batches, the linear term on a coalesced sweep of the row.
//
// The pairwise term is accumulated WITHOUT the reference's cancellation 1/2 (S_f^2 - Q_f)
// (src/core/Model.h:144-158): P_f += t * S_f before S_f += t gives sum_{i<j} t_i t_j directly, and the cross terms
// between sub-groups are S_a * S_b at every combine stage.  Same number of instructions, and fp32 stays within
// 1e-5 of the fp64 reference for any k.
//
// Returns this lane's share of  lin + sum_f P_f  (with_pair), or of the ADDITIVE part
// lin + sum_f P_f - 1/2 sum_f S_f^2  of a column slice (!with_pair: 1/2 sum_f S_f^2 is formed after the slices'
// S_f have been summed); the caller sums it over the team (team_sum).  On return S[ch][i] is the complete S_f for factor
// (ch*LPR + l)*VN + i in every sub-group of the team.
template <class T, int LPR, int CH, int TEAM, int U>
__device__ __forceinline__ T team_gather(const uint32_t* __restrict__ col, const float* __restrict__ val, uint32_t b,
                                         uint32_t e, const T* __restrict__ w, const T* __restrict__ v, int kp, int k1,
                                         bool with_pair, T (&S)[CH][Vec<T>::N])
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NG = TEAM / LPR;
  const int tl = (threadIdx.x & 31) % TEAM;
  const int sg = tl / LPR, l = tl % LPR;

#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
    for (int i = 0; i < VN; ++i) S[ch][i] = T(0);
  T P[VN];
#pragma unroll
  for (int i = 0; i < VN; ++i) P[i] = T(0);
  T lin = T(0);
  if (k1) {
#pragma unroll 1
    for (uint32_t j = b + tl; j < e; j += TEAM) lin += w[__ldg(col + j)] * T(__ldg(val + j));
  }

  const T* vl = v + l * VN;
  const uint32_t rowb = (uint32_t)kp * (uint32_t)sizeof(T);
  uint32_t base = b;
  for (; base + U * NG <= e; base += U * NG) {                 // full batches: no predicates
    const uint32_t* cp = col + base + sg;
    const float* xp = val + base + sg;
    T x[U];
    uint32_t c[U];
    V16 vv[U][CH];
#pragma unroll
    for (int u = 0; u < U; ++u) c[u] = ld_nc_u32(cp + u * NG);
#pragma unroll
    for (int u = 0; u < U; ++u) x[u] = T(ld_nc_f32(xp + u * NG));
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const V16* vr = reinterpret_cast<const V16*>(reinterpret_cast<const char*>(vl) + (uint64_t)c[u] * rowb);
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) vv[u][ch] = ld_nc_v16(vr + ch * LPR);
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        T a[VN];
        vec_to_arr(vv[u][ch], a);
#pragma unroll
        for (int i = 0; i < VN; ++i) {
          const T t = a[i] * x[u];
          P[i] += t * S[ch][i];
          S[ch][i] += t;
        }
      }
  }
  if (base < e) {                                              // tail: predicated
    const uint32_t rem = e - base;                             // 1 .. U*NG - 1
    const uint32_t* cp = col + base + sg;
    const float* xp = val + base + sg;
    T x[U];
    uint32_t c[U];
    V16 vv[U][CH];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool ok = (uint32_t)(u * NG + sg) < rem;
      c[u] = 0u; x[u] = T(0);
      if (ok) { c[u] = ld_nc_u32(cp + u * NG); x[u] = T(ld_nc_f32(xp + u * NG)); }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool ok = (uint32_t)(u * NG + sg) < rem;
      const V16* vr = reinterpret_cast<const V16*>(reinterpret_cast<const char*>(vl) + (uint64_t)c[u] * rowb);
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        memset(&vv[u][ch], 0, sizeof(V16));
        if (ok) vv[u][ch] = ld_nc_v16(vr + ch * LPR);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        T a[VN];
        vec_to_arr(vv[u][ch], a);
#pragma unroll
        for (int i = 0; i < VN; ++i) {
          const T t = a[i] * x[u];
          P[i] += t * S[ch][i];
          S[ch][i] += t;
        }
      }
  }
  // combine the sub-groups: partners a, b add 1/2^(stage+1) S_a S_b each (2^(stage+1) lanes hold the same product)
  T wgt = T(0.5);
#pragma unroll
  for (int o = LPR; o < TEAM; o <<= 1) {
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int i = 0; i < VN; ++i) {
        const T other = __shfl_xor_sync(0xffffffffu, S[ch][i], o);
        P[i] += wgt * (S[ch][i] * other);
        S[ch][i] += other;
      }
    wgt *= T(0.5);
  }
  T part = lin;
#pragma unroll
  for (int i = 0; i < VN; ++i) part += P[i];
  if (!with_pair && sg == 0) {
    T sq = T(0);
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int i = 0; i < VN; ++i) sq += S[ch][i] * S[ch][i];
    part -= T(0.5) * sq;
  }
  return part;
}

template <class T, int TEAM>
__device__ __forceinline__ T team_sum(T x)
{
#pragma unroll
  for (int o = TEAM / 2; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

constexpr int FWD_BLOCKS = 4;      // resident CTAs per SM of the row-forward kernels
// factor rows in flight per sub-group: 8 for warp teams over 16 or 32 lanes per row, otherwise 4
template <int LPR, int TEAM = 32> struct GatherDepth { enum { U = (TEAM == 32 && LPR >= 16) ? 8 : 4 }; };

// score (no link) of the team's row, identical in every lane of the team
template <class T, int LPR, int CH, int TEAM>
__device__ __forceinline__ T team_forward(const uint32_t* __restrict__ col, const float* __restrict__ val, uint32_t b,
                                          uint32_t e, const T* __restrict__ w, const T* __restrict__ v, int kp, T w0,
                                          int k0, int k1, T (&S)[CH][Vec<T>::N])
{
  const T part = team_gather<T, LPR, CH, TEAM, GatherDepth<LPR, TEAM>::U>(col, val, b, e, w, v, kp, k1, true, S);
  return (k0 ? w0 : T(0)) + team_sum<T, TEAM>(part);
}

// column-slice variant: S_f of the slice plus the ADDITIVE part of the score (linear term - 1/2 sum Q);
// 1/2 sum_f S_f^2 is formed after the partial S_f have been summed over the shards
template <class T, int LPR, int CH, int TEAM>
__device__ __forceinline__ T team_forward_partial(const uint32_t* __restrict__ col, const float* __restrict__ val,
                                                  uint32_t b, uint32_t e, const T* __restrict__ w,
                                                  const T* __restrict__ v, int kp, int k1, T (&S)[CH][Vec<T>::N])
{
  const T part = team_gather<T, LPR, CH, TEAM, GatherDepth<LPR, TEAM>::U>(col, val, b, e, w, v, kp, k1, false, S);
  return team_sum<T, TEAM>(part);
}

// rows with at most this many non-zeros per LPR-lane group on average go one row per group
__host__ __device__ inline bool short_rows(int64_t nnz, int64_t n, int lpr) { return lpr < 32 && n > 0 && nnz <= n * 4 * (32 / lpr); }
// 1: one row per LPR-lane group; 2: one row per half warp (two sub-groups; the per-row fixed cost -- bounds, linear sweep,
// combine, team sum, stores -- is shared by two rows per warp); 0: one row per warp.
inline int team_mode(int64_t nnz, int64_t n, int lpr)
{
  if (short_rows(nnz, n, lpr)) return 1;
  // long rows: half-warp teams measured best for every k <= 32 (predict 8.4 -> 6.6 ms at k = 32, 4.8 -> 3.7 ms at k = 8); k = 64 is
  // DRAM-bound either way and keeps one row per 16-lane group
  return lpr <= 8 ? 2 : (lpr == 16 ? 1 : 0);
}

// table-exact fast_pnorm (reference src/util/Random.h:95-111; Y table regenerated, see link_tables.cu)
__device__ __forceinline__ double dev_fast_pnorm(const double* __restrict__ Y, double x)
{
  const double HINV = 549.966731401936, XMAX = 5.20031455849973;
  const double ax = x < 0 ? -x : x;
  double res;
  if (ax > XMAX) {
    res = 0.999999900524235;
  } else {
    const int i = (int)(ax * HINV);
    const double wgt = (ax - (double)i / HINV) * HINV;
    res = wgt * Y[i + 1] + (1.0 - wgt) * Y[i];
  }
  return (ax == x) ? res : 1.0 - res;
}

// table-exact fast_dpnorm = phi(x)/(1-Phi(x)) (reference src/util/Random.h:114-124)
__device__ __forceinline__ double dev_fast_dpnorm(const double* __restrict__ Y, double x)
{
  const double ax = x < 0 ? -x : x;
  if (x < -3.0) return 0.0;
  if (x > 5.0) return 0.1943369 + 0.9754752 * x + 0.4136861 * sqrt(ax) - 0.5034295 * log(ax + 1e-07);
  const int i = (int)((x + 3.0) * 5000);
  const double xi = rint((-3.0 + 2e-4 * (double)i) * 1e4) / 1e4;
  const double wgt = (x - xi) * 5000;
  return wgt * Y[i + 1] + (1.0 - wgt) * Y[i];
}

__device__ __forceinline__ double apply_link(int link, double s, double lo, double hi, const double* __restrict__ pnY)
{
  switch (link) {
    case FMWR_LINK_LOGISTIC: return 1.0 / (1.0 + exp(-s));
    case FMWR_LINK_PROBIT_TABLE: return dev_fast_pnorm(pnY, s);
    case FMWR_LINK_CLAMP: return s < lo ? lo : (s > hi ? hi : s);
    default: return s;
  }
}

// calculate_grad_mult (reference src/solver/SGD_Learner.h:180-191 and twins)
template <class T>
__device__ __forceinline__ T grad_mult(int task, T y_hat, T y, T lo, T hi)
{
  if (task == FMWR_REGRESSION) {
    y_hat = fmin(hi, y_hat);
    y_hat = fmax(lo, y_hat);
    return -(y - y_hat);
  }
  return -y * (T(1) - T(1) / (T(1) + exp(-y * y_hat)));
}
// throughput (minibatch) mode, fp32: MUFU exp / rcp (about 2 ulp) -- the forward kernel is issue-bound
__device__ __forceinline__ float grad_mult_fast(int task, float y_hat, float y, float lo, float hi)
{
  if (task == FMWR_REGRESSION) return -(y - fmaxf(lo, fminf(hi, y_hat)));
  return -y * (1.f - __fdividef(1.f, 1.f + __expf(-y * y_hat)));
}
__device__ __forceinline__ double grad_mult_fast(int task, double y_hat, double y, double lo, double hi) { return grad_mult<double>(task, y_hat, y, lo, hi); }

// dispatch helper: calls F.template run<T, LPR, CH>() for the model's layout
template <class T, class F>
static inline void dispatch_layout(int kp, F&& f)
{
  const int units = kp / Vec<T>::N;
  switch (units) {
    case 1: f.template run<T, 1, 1>(); break;
    case 2: f.template run<T, 2, 1>(); break;
    case 4: f.template run<T, 4, 1>(); break;
    case 8: f.template run<T, 8, 1>(); break;
    case 16: f.template run<T, 16, 1>(); break;
    case 32: f.template run<T, 32, 1>(); break;
    case 64: f.template run<T, 32, 2>(); break;
    case 128: f.template run<T, 32, 4>(); break;
    default: throw Error(FMWR_ERR_UNSUPPORTED, "unsupported padded factor count");
  }
}

}  // namespace fmwr
