// Per-feature contributions of the FM score (fmwr_contrib_dev): the exact Shapley values of the game
// v(T) = score of the row with every entry outside T set to 0.  A pairwise term gives half of its interaction to each of its two
// features, so for entry j of a row
//   phi_j = [k1] w_j x_j + 1/2 x_j sum_f v_jf (S_f - x_j v_jf),   S_f = sum_l v_lf x_l,   and   [k0] w0 + sum_j phi_j = score.
// Pass 1 is the forward's team_gather (score and the complete S_f in every sub-group of the team); pass 2 walks the row's entries
// again, split over the sub-groups the same way, and re-reads each factor row (L1/L2-resident since pass 1) to form phi_j.
#include "forward.cuh"

namespace fmwr {

// resident CTAs per SM: the forward's, except for warp teams over 16 or 32 lanes (8 factor rows in flight in pass 1), which keep
// S_f live through pass 2 and spill under a 64- or 80-register bound
template <int LPR, int TEAM> struct ContribBlocks { enum { N = (TEAM == 32 && LPR >= 16) ? 2 : FWD_BLOCKS }; };

// One batch of pass 2: entries base + u*NG + sg (u < U) of the sub-group, all loads issued before any is consumed.  TAIL: only
// the first rem entries of the batch exist.  The LPR lanes of a group each hold a 16-byte slice of the factor row, reduce their
// partial sums with xor shuffles, and lane u % LPR stores entry u.
template <class T, int LPR, int CH, int TEAM, int U, bool TAIL>
__device__ __forceinline__ void contrib_batch(const uint32_t* __restrict__ col, const float* __restrict__ val, uint32_t base,
                                              uint32_t rem, const T* __restrict__ w, const T* __restrict__ vl, uint32_t rowb,
                                              int k1, unsigned gmask, const T (&S)[CH][Vec<T>::N], double* __restrict__ out)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NG = TEAM / LPR;
  const int tl = (threadIdx.x & 31) % TEAM;
  const int sg = tl / LPR, l = tl % LPR;
  const uint32_t* cp = col + base + sg;
  const float* xp = val + base + sg;
  uint32_t c[U];
  T x[U], wj[U];
  V16 vv[U][CH];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const bool ok = !TAIL || (uint32_t)(u * NG + sg) < rem;
    c[u] = 0u; x[u] = T(0);
    if (ok) { c[u] = ld_nc_u32(cp + u * NG); x[u] = T(ld_nc_f32(xp + u * NG)); }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const bool ok = !TAIL || (uint32_t)(u * NG + sg) < rem;
    const V16* vr = reinterpret_cast<const V16*>(reinterpret_cast<const char*>(vl) + (uint64_t)c[u] * rowb);
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      memset(&vv[u][ch], 0, sizeof(V16));
      if (ok) vv[u][ch] = ld_nc_v16(vr + ch * LPR);
    }
    wj[u] = T(0);
    if (k1 && ok && u % LPR == l) wj[u] = w[c[u]];
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    T part = T(0);
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      T a[VN];
      vec_to_arr(vv[u][ch], a);
#pragma unroll
      for (int i = 0; i < VN; ++i) part += a[i] * (S[ch][i] - x[u] * a[i]);
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) part += __shfl_xor_sync(gmask, part, o);
    const bool ok = !TAIL || (uint32_t)(u * NG + sg) < rem;
    if (ok && u % LPR == l) out[base + u * NG + sg] = (double)(wj[u] * x[u] + T(0.5) * x[u] * part);
  }
}

template <class T, int LPR, int CH, int TEAM>
__global__ void __launch_bounds__(256, ContribBlocks<LPR, TEAM>::N)
contrib_kernel(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
               const T* __restrict__ w, const T* __restrict__ v, const double* __restrict__ scal, int kp, int k0, int k1,
               int64_t n, double* __restrict__ score, double* __restrict__ phi)
{
  constexpr int TPW = 32 / TEAM;           // rows per warp per iteration
  constexpr int NG = TEAM / LPR;
  constexpr int U = GatherDepth<LPR, TEAM>::U / CH;   // pass 2 holds S as well: as many factor-row registers in flight as CH = 1
  const int lane = threadIdx.x & 31;
  const int team = lane / TEAM, tl = lane % TEAM;
  const unsigned gmask = LPR == 32 ? 0xffffffffu : ((1u << LPR) - 1u) << (lane & ~(LPR - 1));
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t step = (int64_t)gridDim.x * (blockDim.x >> 5) * TPW;
  const T w0 = T(scal[0]);
  const T* vl = v + (tl % LPR) * Vec<T>::N;
  const uint32_t rowb = (uint32_t)kp * (uint32_t)sizeof(T);
  for (int64_t base_row = warp0 * TPW; base_row < n; base_row += step) {
    const int64_t row = base_row + team;
    uint32_t b = 0u, e = 0u;
    if (row < n) { b = __ldg(rowptr + row); e = __ldg(rowptr + row + 1); }
    T S[CH][Vec<T>::N];
    const T sc = team_forward<T, LPR, CH, TEAM>(col, val, b, e, w, v, kp, w0, k0, k1, S);
    if (tl == 0 && row < n) score[row] = (double)sc;
    uint32_t base = b;
    for (; base + U * NG <= e; base += U * NG)                 // full batches: no predicates
      contrib_batch<T, LPR, CH, TEAM, U, false>(col, val, base, 0u, w, vl, rowb, k1, gmask, S, phi);
    if (base < e) contrib_batch<T, LPR, CH, TEAM, U, true>(col, val, base, e - base, w, vl, rowb, k1, gmask, S, phi);
  }
}

struct ContribLaunch {
  fmwr_ctx* ctx; fmwr_model* m; fmwr_data* d;
  template <class T, int LPR, int CH>
  void run()
  {
    const int tm = team_mode(d->nnz, d->n, LPR);
    if (tm == 1) go<T, LPR, CH, LPR>();
    else if (tm == 2) go<T, LPR, CH, (LPR <= 8 ? 16 : 32)>();
    else go<T, LPR, CH, 32>();
  }
  template <class T, int LPR, int CH, int TEAM>
  void go()
  {
    const int block = 256, rpb = (block / 32) * (32 / TEAM);
    int64_t want = ceil_div64(d->n, rpb);
    int64_t cap = (int64_t)ctx->sm_count * 32;   // as the forward: 32 CTAs per SM, grid-stride beyond that
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    FMWR_LAUNCH(ctx, (contrib_kernel<T, LPR, CH, TEAM>), grid, block, 0,
                d->rowptr.p, d->col.p, d->val.p, (const T*)m->w.p, (const T*)m->v.p, (const double*)m->scal.p,
                m->kp, m->cfg.keep_w0, m->cfg.keep_w1, d->n, d->pred64.p, d->contrib64.p);
  }
};

void contrib_launch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d)
{
  require_same_features(m, d);
  d->pred64.ensure(d->n);
  d->pred_prec = FMWR_F64;
  if (!d->contrib64.p) d->contrib64.alloc(d->nnz);
  if (d->n == 0) return;
  ContribLaunch f{ctx, m, d};
  if (m->prec == FMWR_F64) dispatch_layout<double>(m->kp, f);
  else dispatch_layout<float>(m->kp, f);
}

}  // namespace fmwr
