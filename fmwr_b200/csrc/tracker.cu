// The tracker of all three trainers (common.cuh: Tracker; reference src/core/Tracker.h, src/solver/SGD_Learner.h:140-175)
#include "common.cuh"

#include <algorithm>
#include <cmath>

namespace fmwr {

// Model::predict_prob (reference src/core/Model.h:163-180): the tracker's link for (task, solver)
int tracker_link(int task, int solver)
{
  if (task == FMWR_REGRESSION) return FMWR_LINK_CLAMP;
  return (solver == FMWR_MCMC || solver == FMWR_ALS) ? FMWR_LINK_PROBIT_TABLE : FMWR_LINK_LOGISTIC;
}

// train-set score for the tracker (reference src/solver/SGD_Learner.h:140-156)
double tracker_score(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s)
{
  forward_launch(ctx, m, d, tracker_link(m->cfg.task, s->solver), s->min_target, s->max_target);
  return evaluate_dev(ctx, d, m->cfg.task, s->metric);
}

// Tracker::init step-size rule (reference src/core/Tracker.h:41-52, MAX_REC = 10000)
static int tracker_step_size(int step_size, int max_iter)
{
  if (step_size <= 0) return step_size;
  const int rt = (int)(std::ceil(((double)max_iter - 0.5) / (double)step_size)) + 1;
  if (rt > 10000) step_size = (int)((double)(max_iter + 1) / 10000.0) + 1;
  return step_size;
}

Tracker::Tracker(fmwr_ctx* ctx_, fmwr_model* m_, const fmwr_solver_cfg* s_, fmwr_trace* tr_, const Holdout* h_)
    : step(tracker_step_size(s_->step_size, s_->max_iter)), ctx(ctx_), m(m_), s(s_), tr(tr_), h(h_) {}

bool Tracker::due_after_batch(int64_t iter)
{
  if (step <= 0 || !(iter > next_track || iter >= s->max_iter)) return false;
  next_track = (iter / step + 1) * (int64_t)step;
  return true;
}

bool Tracker::record(int64_t idx, double score)
{
  const bool converges = s->solver != FMWR_ALS && s->solver != FMWR_MCMC;     // ALS/MCMC report convergent = 0
  if (converges && n_rec >= 2 && std::fabs((score - old_score) / (old_score + 1e-30)) <= s->convergence) conv_times++;
  else conv_times = 0;
  old_score = score;
  if (tr && n_rec < tr->max_rec) {              // records past max_rec count but are not stored
    if (tr->eval_train) tr->eval_train[n_rec] = score;
    if (tr->rec_index) tr->rec_index[n_rec] = (int)idx;
    if (tr->snap_w0 || tr->snap_w || tr->snap_v) {
      double w0 = 0;
      model_get_host(m, &w0, tr->snap_w ? tr->snap_w + (size_t)n_rec * m->p : nullptr,
                     tr->snap_v ? tr->snap_v + (size_t)n_rec * m->p * m->k : nullptr);
      if (tr->snap_w0) tr->snap_w0[n_rec] = w0;
    }
  }
  const bool patience_stop = h && record_holdout();
  n_rec++;
  if (conv_times >= 3) { convergent = 1; return true; }
  return patience_stop;
}

// Held-out sets are scored exactly as tracker_score scores the training data: same model, link and metric.  Better on eval[0]
// is strictly greater for classification (LL, AUC, ACC) and strictly smaller for regression (evaluate_dev returns RMSE or MAE
// there), so ties keep the earlier record and NaN never wins.  Every record counts, stored or not.
bool Tracker::record_holdout()
{
  double score0 = 0.0;
  for (int i = 0; i < h->n_eval; ++i) {
    const double sc = tracker_score(ctx, m, h->eval[i], s);
    if (i == 0) score0 = sc;
    if (n_rec < h->max_rec) h->scores[(size_t)i * h->max_rec + n_rec] = sc;
  }
  const bool cls = m->cfg.task == FMWR_CLASSIFICATION;
  if (!std::isnan(score0) && (best_rec < 0 || (cls ? score0 > best : score0 < best))) {
    best = score0; best_rec = n_rec; since = 0;
    if (h->select_best) {
      const size_t wb = (size_t)m->p * m->esz(), vb = (size_t)m->p * m->kp * m->esz();
      best_w.alloc(wb); best_v.alloc(vb); best_w0.alloc(1);
      if (wb) FMWR_CUDA(cudaMemcpyAsync(best_w.p, m->w.p, wb, cudaMemcpyDeviceToDevice, ctx->stream));
      if (vb) FMWR_CUDA(cudaMemcpyAsync(best_v.p, m->v.p, vb, cudaMemcpyDeviceToDevice, ctx->stream));
      FMWR_CUDA(cudaMemcpyAsync(best_w0.p, m->scal.p, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    }
  } else {
    since++;
  }
  return h->patience > 0 && since >= h->patience;
}

// the best copy goes back over (w0, w, V) only: scal[1..] and the optimizer state stay as training left them
void Tracker::restore_best()
{
  if (!h) return;
  *h->best_rec = best_rec;
  if (!h->select_best || best_rec < 0) return;
  const size_t wb = (size_t)m->p * m->esz(), vb = (size_t)m->p * m->kp * m->esz();
  if (wb) FMWR_CUDA(cudaMemcpyAsync(m->w.p, best_w.p, wb, cudaMemcpyDeviceToDevice, ctx->stream));
  if (vb) FMWR_CUDA(cudaMemcpyAsync(m->v.p, best_v.p, vb, cudaMemcpyDeviceToDevice, ctx->stream));
  FMWR_CUDA(cudaMemcpyAsync(m->scal.p, best_w0.p, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
}

void Tracker::write_trace(int64_t iters_done)
{
  if (tr) { tr->n_rec = std::min(n_rec, (int)tr->max_rec); tr->convergent = convergent; tr->iters_done = (int)iters_done; }
}

}  // namespace fmwr
