// Drop-in replacement for FMwR's src/FM.cpp: the three Rcpp exports keep their signatures
// (reference src/FM.cpp:7, :177, :218; src/RcppExports.cpp is unchanged) and become thin glue that
// unpacks the R lists into raw pointers and calls libfmwr_b200.so (include/fmwr_b200.h).
//
// Device copies of fm.matrix objects persist across calls (see "persistent handles" below); the default precision is the
// reference's fp64 except in the throughput mode.
//
// UNVERIFIED IN THIS REPOSITORY: the build image has no R / Rcpp, so this file has never been compiled.
// It is the binding a maintainer adds; the same call sequence is exercised by fmwr_b200/api.py.
//
// Build: src/Makevars gains   PKG_CPPFLAGS = -I$(FMWR_B200)/include
//                             PKG_LIBS     = -L$(FMWR_B200)/fmwr_b200 -lfmwr_b200 -Wl,-rpath,$(FMWR_B200)/fmwr_b200
#include <Rcpp.h>
#include <map>
#include <string>
#include <vector>
#include "fmwr_b200.h"

using namespace Rcpp;

static void check(int rc) { if (rc != 0) stop(fmwr_last_error()); }   // Rcpp::stop -> R error, as before

// ---- persistent handles (SURVEY 8f-3) -------------------------------------------------------------------------------------
// The reference deep-copies the fm.matrix lists on every .Call (src/FM.cpp:31-34).  Here the device copy of an fm.matrix is
// created once and parked in an external pointer stored as attribute "fmwr.handle" of its `features` list; R's copy-on-modify
// gives a modified matrix new vectors, so the key (addresses + sizes of value / col_idx / row_size) goes stale exactly when the
// contents can have changed.  The finalizer frees the device memory when R collects the object.  options(FM.cache = FALSE)
// restores upload-per-call.  One context per device lives for the session.
struct Parked {
  fmwr_data* d; const void* kv; const void* kc; const void* kr; R_xlen_t nnz; int n, p; const void* klab;
};
static void parked_finalizer(SEXP xp)
{
  Parked* h = static_cast<Parked*>(R_ExternalPtrAddr(xp));
  if (h) { fmwr_data_destroy(h->d); delete h; R_ClearExternalPtr(xp); }
}
static fmwr_ctx* session_ctx(int device)
{
  static std::map<int, fmwr_ctx*> ctxs;
  if (!ctxs.count(device)) { fmwr_ctx* c = NULL; check(fmwr_ctx_create(device, &c)); ctxs[device] = c; }
  return ctxs[device];
}
static bool opt_flag(const char* name, bool dflt)
{
  Function getOption("getOption");
  return as<bool>(getOption(name, dflt));
}
// device handle of an fm.matrix; `owned` tells the caller to destroy it (caching off).  labels may be R_NilValue (predict).
static fmwr_data* acquire(fmwr_ctx* ctx, List X, SEXP labels, bool will_rescale, bool* owned)
{
  NumericVector value = X["value"]; IntegerVector col_idx = X["col_idx"]; IntegerVector row_size = X["row_size"]; IntegerVector dim = X["dim"];
  const int64_t n = dim[0], p = dim[1], nnz = value.size();
  const double* lab = Rf_isNull(labels) ? NULL : REAL(labels);
  *owned = !opt_flag("FM.cache", true);
  if (!*owned) {
    SEXP slot = X.attr("fmwr.handle");
    if (!Rf_isNull(slot) && TYPEOF(slot) == EXTPTRSXP && R_ExternalPtrAddr(slot)) {
      Parked* h = static_cast<Parked*>(R_ExternalPtrAddr(slot));
      if (h->kv == (const void*)value.begin() && h->kc == (const void*)col_idx.begin() && h->kr == (const void*)row_size.begin() &&
          h->nnz == value.size() && h->n == dim[0] && h->p == dim[1]) {
        if (lab && h->klab != (const void*)lab) { check(fmwr_data_set_labels(h->d, lab)); h->klab = lab; }
        if (!will_rescale) check(fmwr_data_restore_values(h->d));      // fmwr_data_scales / normalize start from the uploaded values themselves
        return h->d;
      }
    }
  }
  fmwr_data* d = NULL;
  check(fmwr_data_create(ctx, n, p, nnz, row_size.begin(), col_idx.begin(), value.begin(), lab, &d));
  if (!*owned) {
    Parked* h = new Parked{d, value.begin(), col_idx.begin(), row_size.begin(), value.size(), dim[0], dim[1], lab};
    SEXP xp = PROTECT(R_MakeExternalPtr(h, R_NilValue, R_NilValue));
    R_RegisterCFinalizerEx(xp, parked_finalizer, TRUE);
    Rf_setAttrib(X, Rf_install("fmwr.handle"), xp);                    // in place: the slot belongs to the caller's object
    UNPROTECT(1);
  }
  return d;
}

// FM.precision: "auto" (default) = fp64 wherever the result is held to the reference's (exact mode, ALS, MCMC, predict),
// fp32 in the throughput (minibatch) mode; "f32" / "f64" force it
static int precision_for(int solver, bool minibatch)
{
  const std::string o = opt_str("FM.precision", "auto");
  if (o == "f64") return FMWR_F64;
  if (o == "f32") return FMWR_F32;
  return (minibatch && (solver == FMWR_SGD || solver == FMWR_FTRL || solver == FMWR_TDAP)) ? FMWR_F32 : FMWR_F64;
}

static int opt_int(const char* name, int dflt)
{
  Function getOption("getOption");
  SEXP v = getOption(name, dflt);
  return as<int>(v);
}

static std::string opt_str(const char* name, const char* dflt)
{
  Function getOption("getOption");
  return as<std::string>(getOption(name, dflt));
}

static fmwr_model_cfg model_cfg(List fm_controls)
{
  std::map<std::string, int> tasks; tasks["CLASSIFICATION"] = FMWR_CLASSIFICATION; tasks["REGRESSION"] = FMWR_REGRESSION;
  List hp = fm_controls["hyper.params"];
  fmwr_model_cfg c;
  c.task = tasks[as<std::string>(fm_controls["task"])];
  c.keep_w0 = (bool)hp["keep.w0"]; c.keep_w1 = (bool)hp["keep.w1"]; c.k = (int)hp["factor.number"];
  c.l2_w0 = (double)hp["L2.w0"]; c.l1_w1 = (double)hp["L1.w1"]; c.l2_w1 = (double)hp["L2.w1"];
  c.l1_v = (double)hp["L1.v"]; c.l2_v = (double)hp["L2.v"];
  return c;
}

static int solver_id(List solver_controls)
{
  std::map<std::string, int> m;
  m["MCMC"] = FMWR_MCMC; m["ALS"] = FMWR_ALS; m["SGD"] = FMWR_SGD; m["FTRL"] = FMWR_FTRL; m["TDAP"] = FMWR_TDAP;
  List solver = solver_controls["solver"];
  std::string s = as<std::string>(solver.attr("solver"));
  if (!m.count(s)) stop("Unknown solver...");
  return m[s];
}

static int metric_id(const std::string& s)
{
  std::map<std::string, int> m;
  m["LL"] = FMWR_LL; m["AUC"] = FMWR_AUC; m["ACC"] = FMWR_ACC; m["RMSE"] = FMWR_RMSE; m["MSE"] = FMWR_MSE; m["MAE"] = FMWR_MAE;
  return m[s];
}

// [[Rcpp::export]]
List FM(List data_, IntegerVector normalize, List fm_controls, List solver_controls, List track_controls, List model_list)
{
  List X = data_["features"];
  NumericVector value = X["value"]; IntegerVector col_idx = X["col_idx"]; IntegerVector row_size = X["row_size"];
  IntegerVector dim = X["dim"];
  NumericVector target = as<NumericVector>(data_["labels"]);
  const int64_t n = dim[0], p = dim[1], nnz = value.size();

  fmwr_ctx* ctx = session_ctx(opt_int("FM.device", 0));
  fmwr_model* m = NULL;
  bool owned = false;
  fmwr_data* d = acquire(ctx, X, target, normalize[0] > -1, &owned);

  List scales;
  if (normalize[0] > -1) {                                            // reference FM.cpp:36-38
    NumericVector mean(p), sd(p);
    check(fmwr_data_scales(d, normalize.begin(), normalize.size(), mean.begin(), sd.begin()));
    scales["mean"] = mean; scales["std"] = sd;
  }
  scales["model.vars"] = as<CharacterVector>(X.attr("feature_names"));

  fmwr_model_cfg mc = model_cfg(fm_controls);
  List hp = fm_controls["hyper.params"];
  const int k = mc.k;
  const bool minibatch = opt_str("FM.mode", "exact") == "minibatch";
  const int prec = precision_for(solver_id(solver_controls), minibatch);
  check(fmwr_model_create(ctx, &mc, p, prec, &m));

  // Model::init (reference src/core/Model.h:63-72): w = 0, V ~ rnorm drawn HERE, factor-major, so set.seed() holds
  double w0 = 0.0;
  NumericVector w(p);
  NumericMatrix v(k, p);                                              // k x p column-major == the engine's [p][k]
  {
    std::vector<double> draws((size_t)k * p);
    for (size_t i = 0; i < draws.size(); ++i) draws[i] = Rf_rnorm((double)hp["v.init_mean"], (double)hp["v.init_stdev"]);
    for (int f = 0; f < k; ++f) for (int64_t j = 0; j < p; ++j) v(f, j) = draws[(size_t)f * p + j];
  }
  double lo = min(target), hi = max(target);
  SEXP is_model = model_list.attr("class");
  if (!Rf_isNull(is_model)) {                                         // warm start (fm.update), FM.cpp:66-72, :91-96
    List model = model_list["Model"];
    w0 = (double)model["w0"]; w = clone(as<NumericVector>(model["w"])); v = clone(as<NumericMatrix>(model["v"]));
    List so = model_list["Scales"];
    NumericVector tr = as<NumericVector>(so.attr("target.range"));
    lo = std::min(lo, tr[0]); hi = std::max(hi, tr[1]);
  }
  check(fmwr_model_set(m, w0, w.begin(), v.begin()));

  List solver = solver_controls["solver"];
  fmwr_solver_cfg sc; memset(&sc, 0, sizeof sc);
  sc.solver = solver_id(solver_controls);
  sc.max_iter = (int)solver_controls["max_iter"];
  sc.random_step = solver.containsElementNamed("random_step") ? (int)solver["random_step"] : 1;
  sc.learn_rate = solver.containsElementNamed("learn_rate") ? (double)solver["learn_rate"] : 0.01;
  sc.alpha_w = solver.containsElementNamed("alpha_w") ? (double)solver["alpha_w"] : 0.1;
  sc.alpha_v = solver.containsElementNamed("alpha_v") ? (double)solver["alpha_v"] : 0.1;
  sc.beta_w = solver.containsElementNamed("beta_w") ? (double)solver["beta_w"] : 1.0;
  sc.beta_v = solver.containsElementNamed("beta_v") ? (double)solver["beta_v"] : 1.0;
  sc.gamma = solver.containsElementNamed("gamma") ? (double)solver["gamma"] : 1e-4;
  sc.min_target = lo; sc.max_target = hi;
  sc.mode = minibatch ? FMWR_MODE_MINIBATCH : FMWR_MODE_EXACT;
  sc.batch_size = opt_int("FM.batch", 65536);
  sc.precision = prec;
  sc.compat = opt_str("FM.compat", "reference") == "reference" ? FMWR_COMPAT_REFERENCE : 0;
  sc.enable_v = opt_int("FM.enable_v", 0);
  sc.step_size = (int)track_controls["step_size"];
  sc.metric = metric_id(as<std::string>(track_controls["evaluate.metric"]));
  sc.convergence = (double)track_controls["convergence"];
  sc.seed = (uint64_t)(R::unif_rand() * 4294967296.0);               // native MCMC RNG keyed off R's stream
  // MCMC attribute groups (libFM's feature grouping): x$features$attr_group <- g, 0-based, one entry per column
  IntegerVector attr_group;
  if (sc.solver == FMWR_MCMC && X.containsElementNamed("attr_group") && !Rf_isNull(X["attr_group"])) {
    attr_group = as<IntegerVector>(X["attr_group"]);
    if (attr_group.size() != p) Rcpp::stop("attr_group must be an integer vector with one entry per column");
    int mx = 0;
    for (int i = 0; i < attr_group.size(); ++i) mx = std::max(mx, (int)attr_group[i]);
    sc.attr_group = attr_group.begin(); sc.n_groups = mx + 1;            // range checks: fmwr_train_dev (FMWR_ERR_ARG)
  }

  fmwr_trace tr; memset(&tr, 0, sizeof tr);
  std::vector<double> ev, sw0, sw, sv; std::vector<int> ri;
  if (sc.step_size > 0) {
    tr.max_rec = std::min(10001, (int)std::ceil((sc.max_iter - 0.5) / sc.step_size) + 2);
    ev.resize(tr.max_rec); ri.resize(tr.max_rec); sw0.resize(tr.max_rec);
    sw.resize((size_t)tr.max_rec * p); sv.resize((size_t)tr.max_rec * p * std::max(k, 1));
    tr.eval_train = ev.data(); tr.rec_index = ri.data(); tr.snap_w0 = sw0.data(); tr.snap_w = sw.data(); tr.snap_v = sv.data();
  }
  int rc = fmwr_train_dev(ctx, m, d, &sc, sc.step_size > 0 ? &tr : NULL);
  if (rc == 0) rc = fmwr_model_get(m, &w0, w.begin(), v.begin());
  fmwr_model_destroy(m);
  if (owned) fmwr_data_destroy(d);
  check(rc);
  const int n_rec = std::min(tr.n_rec, tr.max_rec);                   // records actually written (never read past the buffers)

  List md = List::create(_["w0"] = w0, _["w"] = w, _["v"] = v);      // Model::save_model
  md.attr("model.control") = fm_controls;
  md.attr("solver.control") = solver_controls;
  md.attr("track.control") = track_controls;
  md.attr("convergence") = (bool)tr.convergent;
  List res;
  res["Model"] = md;
  scales.attr("target.range") = NumericVector::create(lo, hi);
  res["Scales"] = scales;
  if (sc.step_size > 0) {                                             // Tracker::save, src/core/Tracker.h:96-119
    List valid(n_rec + 1);
    NumericVector idx(n_rec);
    for (int i = 0; i < n_rec; ++i) idx[i] = ri[i];
    valid[0] = idx;
    for (int i = 0; i < n_rec; ++i) {
      NumericVector wi(sw.begin() + (size_t)i * p, sw.begin() + (size_t)(i + 1) * p);
      NumericMatrix vi(k, p);
      std::copy(sv.begin() + (size_t)i * p * k, sv.begin() + (size_t)(i + 1) * p * k, vi.begin());
      valid[i + 1] = List::create(_["w0"] = sw0[i], _["w"] = wi, _["v"] = vi);
    }
    res["Trace"] = List::create(_["trace"] = valid, _["evaluation.train"] = NumericVector(ev.begin(), ev.begin() + n_rec));
  }
  res.attr("class") = "FM";
  return res;
}

// [[Rcpp::export]]
NumericVector FMPredict(List newdata, bool normalize, List model_list, int max_threads)
{
  List X = newdata["features"];
  IntegerVector dim = X["dim"];
  const int64_t n = dim[0], p = dim[1];
  List model = model_list["Model"];
  List scales = model_list["Scales"];                                 // read unconditionally (latent crash in the reference, SURVEY 3.2)
  fmwr_model_cfg mc = model_cfg(as<List>(model.attr("model.control")));
  const int solver = solver_id(as<List>(model.attr("solver.control")));
  const int prec = precision_for(0, false);
  NumericVector w = model["w"]; NumericMatrix v = model["v"];
  NumericVector tr = as<NumericVector>(scales.attr("target.range"));

  fmwr_ctx* ctx = session_ctx(opt_int("FM.device", 0));
  fmwr_model* m = NULL;
  bool owned = false;
  fmwr_data* d = acquire(ctx, X, R_NilValue, normalize, &owned);
  if (normalize) {
    NumericVector mean = scales["mean"], sd = scales["std"];
    check(fmwr_data_normalize(d, mean.begin(), sd.begin()));
  }
  check(fmwr_model_create(ctx, &mc, p, prec, &m));
  check(fmwr_model_set(m, (double)model["w0"], w.begin(), v.begin()));
  int link = mc.task == FMWR_CLASSIFICATION
                 ? ((solver == FMWR_MCMC || solver == FMWR_ALS) ? FMWR_LINK_PROBIT_TABLE : FMWR_LINK_LOGISTIC)
                 : FMWR_LINK_CLAMP;                                   // Model::predict_prob / FM.cpp:204-210
  NumericVector pred(n);
  int rc = fmwr_predict_dev(ctx, m, d, link, tr[0], tr[1]);
  if (rc == 0) rc = fmwr_predict_fetch(ctx, d, pred.begin());
  fmwr_model_destroy(m);
  if (owned) fmwr_data_destroy(d);
  check(rc);
  return pred;
}

// [[Rcpp::export]]
NumericVector FMTrack(List newdata, List model_list, bool normalize, String type, int max_threads)
{
  // Tracker::report (src/core/Tracker.h:70-94): per recorded snapshot a forward over newdata + the metric, on the parked handle
  List X = newdata["features"];
  IntegerVector dim = X["dim"];
  const int64_t p = dim[1];
  List model = model_list["Model"]; List scales = model_list["Scales"];
  fmwr_model_cfg mc = model_cfg(as<List>(model.attr("model.control")));
  const int solver = solver_id(as<List>(model.attr("solver.control")));
  NumericVector tr = as<NumericVector>(scales.attr("target.range"));
  fmwr_ctx* ctx = session_ctx(opt_int("FM.device", 0));
  bool owned = false;
  fmwr_data* d = acquire(ctx, X, newdata["labels"], normalize, &owned);
  if (normalize) {                                                    // SMatrix::normalize, Smatrix.h:144-150
    NumericVector mean = scales["mean"], sd = scales["std"];
    check(fmwr_data_normalize(d, mean.begin(), sd.begin()));
  }
  fmwr_model* m = NULL;
  check(fmwr_model_create(ctx, &mc, p, precision_for(0, false), &m));
  const int link = mc.task == FMWR_CLASSIFICATION
                       ? ((solver == FMWR_MCMC || solver == FMWR_ALS) ? FMWR_LINK_PROBIT_TABLE : FMWR_LINK_LOGISTIC)
                       : FMWR_LINK_CLAMP;
  List trace = model_list["Trace"]; List snaps = trace["trace"];
  const int ns = snaps.size() - 1;
  NumericVector out(ns);
  int rc = 0;
  for (int i = 0; i < ns && rc == 0; ++i) {
    List s = snaps[i + 1];
    NumericVector wi = s["w"]; NumericMatrix vi = s["v"];
    rc = fmwr_model_set(m, (double)s["w0"], wi.begin(), vi.begin());
    if (rc == 0) rc = fmwr_predict_dev(ctx, m, d, link, tr[0], tr[1]);
    if (rc == 0) rc = fmwr_evaluate_dev(ctx, d, mc.task, metric_id(type), &out[i]);
  }
  fmwr_model_destroy(m);
  if (owned) fmwr_data_destroy(d);
  check(rc);
  return out;
}
