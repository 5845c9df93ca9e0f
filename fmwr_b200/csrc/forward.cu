// predict.FM / error-cache forward pass: replaces Model::predict_batch + predict_prob + the
// regression clamp (reference src/core/Model.h:106-180, src/FM.cpp:197-211).
#include "forward_stream.cuh"

#include <algorithm>
namespace fmwr {

template <class T, int LPR, int CH, int TEAM>
__global__ void __launch_bounds__(256, FWD_BLOCKS)
forward_kernel(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
               const T* __restrict__ w, const T* __restrict__ v, const double* __restrict__ scal, int kp, int k0, int k1,
               int64_t n, int link, double lo, double hi, const double* __restrict__ pnY, double* __restrict__ out)
{
  constexpr int TPW = 32 / TEAM;           // rows per warp per iteration
  constexpr int SLOTS = 32 / TPW;          // iterations between two link flushes
  const int lane = threadIdx.x & 31;
  const int team = lane / TEAM;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t step = (int64_t)gridDim.x * (blockDim.x >> 5) * TPW;
  const T w0 = T(scal[0]);
  // The link function runs in fp64 (see FwdLaunch) -- ~150 issue slots if done per row by one lane.  Instead lane L
  // parks the score of the (L % TPW)-th row of iteration slot L / TPW and all 32 lanes apply the link together.
  double pending = 0.0;
  int slot = 0;
  int64_t flush_base = warp0 * TPW;
  auto flush = [&](int filled) {
    const int64_t r = flush_base + (int64_t)(lane / TPW) * step + (lane % TPW);
    if (lane / TPW < filled && r < n) out[r] = apply_link(link, pending, lo, hi, pnY);
  };
  for (int64_t base_row = warp0 * TPW; base_row < n; base_row += step) {
    const int64_t row = base_row + team;
    uint32_t b = 0u, e = 0u;
    if (row < n) { b = __ldg(rowptr + row); e = __ldg(rowptr + row + 1); }
    T S[CH][Vec<T>::N];
    const T score = team_forward<T, LPR, CH, TEAM>(col, val, b, e, w, v, kp, w0, k0, k1, S);
    const T sc = (TPW == 1) ? score : __shfl_sync(0xffffffffu, score, (lane % TPW) * TEAM);
    if (slot == lane / TPW) pending = (double)sc;
    if (++slot == SLOTS) { flush(SLOTS); slot = 0; flush_base = base_row + step; }
  }
  if (slot > 0) flush(slot);
}

struct FwdLaunch {
  fmwr_ctx* ctx; fmwr_model* m; fmwr_data* d; int link; double lo, hi;
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
    int64_t cap = (int64_t)ctx->sm_count * 32;   // 32 CTAs per SM, grid-stride beyond that
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    // predictions are always kept in fp64 (8 of ~5.5 KB per row): the R side wants a NumericVector and the
    // reference's log-likelihood (src/core/Evaluation.h:80-89) is NaN for a probability rounded to exactly 1.0f
    d->pred64.ensure(d->n);
    double* out = d->pred64.p;
    d->pred_prec = FMWR_F64;
    FMWR_LAUNCH(ctx, (forward_kernel<T, LPR, CH, TEAM>), grid, block, 0,
                d->rowptr.p, d->col.p, d->val.p, (const T*)m->w.p, (const T*)m->v.p, (const double*)m->scal.p,
                m->kp, m->cfg.keep_w0, m->cfg.keep_w1, d->n, link, lo, hi, ctx->pn_table.p, out);
  }
};

void forward_launch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, int link, double lo, double hi)
{
  // shape checks of Model::predict_batch (reference src/core/Model.h:112-113)
  FMWR_REQUIRE(d->p == m->p, FMWR_ERR_SHAPE, "number of input's features is not correct...");
  if (d->n == 0) return;
  if (stream_forward_ok(m, d->nnz, d->n)) {
    // fp32, 32-float factor rows, long rows: the software-pipelined stream kernel (forward_stream.cuh) + elementwise link
    d->pred64.ensure(d->n);
    d->pred_prec = FMWR_F64;
    SfArgs a;
    memset(&a, 0, sizeof a);
    a.rowptr = d->rowptr.p; a.col = d->col.p; a.val = d->val.p; a.w = (const float*)m->w.p; a.v = (const float*)m->v.p;
    a.scal = (const double*)m->scal.p; a.k0 = m->cfg.keep_w0; a.k1 = m->cfg.keep_w1; a.row_begin = 0; a.rows = d->n; a.out = d->pred64.p;
    const int grid = stream_grid(ctx, d->n, &a.rpg);
    FMWR_LAUNCH(ctx, forward_stream_kernel<SF_PREDICT>, grid, 256, 0, a);
    if (link != FMWR_LINK_NONE) FMWR_LAUNCH(ctx, link_inplace_kernel, ceil_div(d->n, 256), 256, 0, d->pred64.p, d->n, link, lo, hi, ctx->pn_table.p);
    return;
  }
  FwdLaunch f{ctx, m, d, link, lo, hi};
  if (m->prec == FMWR_F64) dispatch_layout<double>(m->kp, f);
  else dispatch_layout<float>(m->kp, f);
}

}  // namespace fmwr
