// SGDA: exact (batch = 1) SGD that learns its L2 rates on a validation set while it trains (Rendle, "Learning recommender
// systems with adaptive regularization", WSDM 2012; libFM's -method sgda).  The rules are in include/fmwr_b200.h
// (fmwr_train_sgda_dev), the two formulas in coord.cuh (sgda_step, sgda_v_term, sgda_lambda_step).
//
// Sample t is a training row's theta step followed, from the second pass on, by one validation row's lambda step, and each
// sample depends on the one before (theta feeds lambda feeds theta), so one persistent CTA walks the samples with the roles of
// exact_kernel (train_exact.cu), which serves the SGD / FTRL / TDAP steps and is left as it is:
//   * factor warps: thread (slot, l) owns non-zero `slot` of a row (rounds of SLOTS for longer rows) and 16-byte vector l of
//     that feature's factor row;
//   * the linear warp: lane = non-zero, owns w_j, its gradient and the row's groups;
//   * the pipeline warp: stages sample t+1's two rows (bounds, label, columns, values, groups) into shared memory by sample
//     parity, prefetches their theta, gradient and lambda lines into L2, sums S_f and the multiplier, and owns w0.
// Per sample: forward (barrier) multiplier (barrier) theta step (barrier), then for the lambda step: look-ahead forward
// (barrier) multiplier (barrier) per-entry terms (barrier) per-group sums and lambda (barrier).  The per-group sums have a fixed
// order and no atomics: the first entry of a group in the row (its leader) sums the group's terms in row order.
#include "forward.cuh"
#include "coord.cuh"

#include <cmath>
#include <vector>

namespace fmwr {

constexpr int SA_THREADS = 512;
constexpr int SA_FW = SA_THREADS / 32 - 2;   // factor warps

template <class T>
struct SgdaArgs {
  const uint32_t* rowptr; const uint32_t* col; const float* val; const float* y;        // training rows
  const uint32_t* vrowptr; const uint32_t* vcol; const float* vval; const float* vy;    // validation rows
  const uint16_t* grp;       // [p] attribute group of each feature
  T* w; T* v; double* scal;
  T* gw; T* gv;              // last gradient of every coordinate, [p] and [p][kp] (zero until a training row touches it)
  double* lam_w; double* lam_v;   // [G] and [G][kp]
  double* cv; double* cw; uint32_t* cg;   // the validation row's per-entry terms [nnz][kp] and [nnz], and groups [nnz]
  int kp, k0, k1, task;
  int64_t n_val;
  const uint32_t* order;     // explicit visit order (NULL: scan)
  int skip_row0;             // F5: scan rows 1..n-1
  int64_t period;            // length of the visit sequence the samples cycle through
  int64_t t0;                // T0, the samples of its first pass: lambda steps start at sample t0
  double lr;                 // learn_rate in fp64, for the fp64 lambda steps
  int64_t t_begin, t_end;    // sample counters of this launch
  SolverParams<T> sp;
  double lo, hi;
};

__device__ __forceinline__ void sa_bar() { asm volatile("bar.sync 0;" ::: "memory"); }

template <class T, int LPR, int CH>
__global__ void __launch_bounds__(SA_THREADS, 1) sgda_kernel(SgdaArgs<T> a)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int SLOTS = SA_FW * 32 / LPR;
  constexpr int SPW = 32 / LPR;              // slots per factor warp
  constexpr int RN = SLOTS > 64 ? SLOTS : 64;   // non-zeros of a row staged in shared memory
  constexpr int NC = (RN + 31) / 32;
  constexpr int W_PIPE = SA_FW, W_LIN = SA_FW + 1;
  constexpr int LINE = 128 / (int)sizeof(T);
  __shared__ V16 sS[SA_FW][LPR * CH];
  __shared__ T sPart[SA_FW];
  __shared__ T sLin;
  __shared__ V16 sSf[LPR * CH];
  __shared__ T sMult;
  __shared__ double sW0;
  // [sample parity][0: training row, 1: validation row]
  __shared__ uint32_t rB[2][2], rE[2][2];
  __shared__ float rY[2][2];
  __shared__ uint32_t rCol[2][2][RN];
  __shared__ float rVal[2][2][RN];
  __shared__ uint16_t rGrp[2][2][RN];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = tid / LPR, l = tid % LPR;
  const int kp = a.kp;
  const T lr = a.sp.lr;
  if (a.t_begin >= a.t_end) return;

  // pipeline warp: sample s's rows into the rings of parity s & 1, their parameter, gradient and lambda lines into L2
  auto stage = [&](int64_t s) {
    const int par = (int)(s & 1);
    const int64_t q = s % a.period;
    const uint32_t r = a.order ? a.order[q] : (uint32_t)(a.skip_row0 ? q + 1 : q);
    const bool vs = s >= a.t0;
    const uint32_t u = vs ? (uint32_t)((s - a.t0) % a.n_val) : 0u;
    uint32_t b[2], e[2];
    b[0] = a.rowptr[r]; e[0] = a.rowptr[r + 1];
    b[1] = vs ? a.vrowptr[u] : 0u; e[1] = vs ? a.vrowptr[u + 1] : 0u;
    if (lane == 0) {
      rB[par][0] = b[0]; rE[par][0] = e[0]; rY[par][0] = a.y[r];
      rB[par][1] = b[1]; rE[par][1] = e[1]; rY[par][1] = vs ? a.vy[u] : 0.f;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t* colp = h ? a.vcol : a.col;
      const float* valp = h ? a.vval : a.val;
#pragma unroll
      for (int c8 = 0; c8 < NC; ++c8) {
        const uint32_t idx = c8 * 32 + lane, j = b[h] + idx;
        if (idx < (uint32_t)RN && j < e[h]) {
          const uint32_t c = colp[j];
          const uint16_t g = a.grp[c];
          rCol[par][h][idx] = c; rVal[par][h][idx] = valp[j]; rGrp[par][h][idx] = g;
          const size_t off = (size_t)c * kp;
          for (int z = 0; z < kp; z += LINE) {
            prefetch_l2(a.v + off + z);
            prefetch_l2(a.gv + off + z);
          }
          for (int z = 0; z < kp; z += 16) prefetch_l2(a.lam_v + (size_t)g * kp + z);
          if (a.k1) { prefetch_l2(a.w + c); prefetch_l2(a.gw + c); prefetch_l2(a.lam_w + g); }
        }
      }
    }
  };

  if (warp == W_PIPE) {
    stage(a.t_begin);
    if (lane == 0) sW0 = a.scal[0];
  }
  __syncthreads();

  // pipeline warp: S_f over the factor warps (lane = factor), the score and its multiplier, published through shared memory
  auto reduce_mult = [&](int nwA, T yv) {
    T acc = T(0);
    T* const sf_out = reinterpret_cast<T*>(sSf);
    for (int f = lane; f < LPR * CH * VN; f += 32) {
      T sf = T(0);
#pragma unroll
      for (int w2 = 0; w2 < SA_FW; ++w2)
        if (w2 < nwA) sf += reinterpret_cast<const T*>(sS[w2])[f];
      sf_out[f] = sf;
      acc += T(0.5) * sf * sf;
    }
    if (lane < nwA) acc += sPart[lane];
    acc = warp_sum(acc);
    acc += sLin;
    const T score = (a.k0 ? T(sW0) : T(0)) + acc;
    if (lane == 0) sMult = grad_mult<T>(a.task, score, yv, T(a.lo), T(a.hi));
  };

  // a row's non-zero i (staged ring for i < RN, global memory beyond)
  auto entry = [&](int par, int h, uint32_t b, uint32_t i, uint32_t& c, T& x, uint32_t& g) {
    if (i < (uint32_t)RN) { c = rCol[par][h][i]; x = T(rVal[par][h][i]); g = rGrp[par][h][i]; }
    else { c = (h ? a.vcol : a.col)[b + i]; x = T((h ? a.vval : a.val)[b + i]); g = a.grp[c]; }
  };

  for (int64_t t = a.t_begin; t < a.t_end; ++t) {
    const int par = (int)(t & 1);
    const bool lam_step = t >= a.t0;         // uniform over the CTA
    // ================= theta step on the training row =================
    {
      const uint32_t b = rB[par][0], e = rE[par][0], nnz = e - b;
      const int nwA = (int)((min(nnz, (uint32_t)SLOTS) + SPW - 1) / SPW);
      if (warp < SA_FW) {
        const bool act = warp < nwA;
        T kth[CH][VN], klam[CH][VN];
        if (act) {
          T S[CH][VN];
          T qsum = T(0);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
#pragma unroll
            for (int i = 0; i < VN; ++i) S[ch][i] = T(0);
          for (uint32_t i0 = 0; i0 < nnz; i0 += SLOTS) {
            const uint32_t i = i0 + slot;
            if (i < nnz) {
              uint32_t c, g; T x;
              entry(par, 0, b, i, c, x, g);
              const V16* vr = reinterpret_cast<const V16*>(a.v + (size_t)c * kp);
#pragma unroll
              for (int ch = 0; ch < CH; ++ch) {
                T arr[VN];
                vec_to_arr(vr[ch * LPR + l], arr);
#pragma unroll
                for (int k = 0; k < VN; ++k) {
                  const T tt = arr[k] * x;
                  S[ch][k] += tt;
                  qsum += tt * tt;
                }
                if (i0 == 0) {
                  const double* lv = a.lam_v + (size_t)g * kp + (ch * LPR + l) * VN;
#pragma unroll
                  for (int k = 0; k < VN; ++k) { kth[ch][k] = arr[k]; klam[ch][k] = T(lv[k]); }
                }
              }
            }
          }
#pragma unroll
          for (int o = LPR; o < 32; o <<= 1)
#pragma unroll
            for (int ch = 0; ch < CH; ++ch)
#pragma unroll
              for (int k = 0; k < VN; ++k) S[ch][k] += __shfl_xor_sync(0xffffffffu, S[ch][k], o);
          const T part = warp_sum(T(-0.5) * qsum);
          if (lane < LPR) {
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) sS[warp][ch * LPR + l] = arr_to_vec(S[ch]);
          }
          if (lane == 0) sPart[warp] = part;
        }
        sa_bar();
        sa_bar();
        if (act) {
          const T mult = sMult;
          T Sf[CH][VN];
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) vec_to_arr(sSf[ch * LPR + l], Sf[ch]);
          for (uint32_t i0 = 0; i0 < nnz; i0 += SLOTS) {
            const uint32_t i = i0 + slot;
            if (i < nnz) {
              uint32_t c, g; T x;
              entry(par, 0, b, i, c, x, g);
              const size_t off = (size_t)c * kp;
              V16* vr = reinterpret_cast<V16*>(a.v + off);
              V16* gr = reinterpret_cast<V16*>(a.gv + off);
#pragma unroll
              for (int ch = 0; ch < CH; ++ch) {
                const int vi = ch * LPR + l;
                T th[VN], lam[VN], gh[VN];
                if (i0 == 0) {
#pragma unroll
                  for (int k = 0; k < VN; ++k) { th[k] = kth[ch][k]; lam[k] = klam[ch][k]; }
                } else {
                  vec_to_arr(vr[vi], th);
                  const double* lv = a.lam_v + (size_t)g * kp + vi * VN;
#pragma unroll
                  for (int k = 0; k < VN; ++k) lam[k] = T(lv[k]);
                }
#pragma unroll
                for (int k = 0; k < VN; ++k) {
                  gh[k] = mult * fm_grad(Sf[ch][k], th[k], x);
                  th[k] = sgda_step(th[k], gh[k], lr, lam[k]);
                }
                gr[vi] = arr_to_vec(gh);
                vr[vi] = arr_to_vec(th);
              }
            }
          }
        }
        sa_bar();
      } else if (warp == W_LIN) {
        T lin = T(0);
        if (a.k1) {
          for (uint32_t i = lane; i < nnz; i += 32) {
            uint32_t c, g; T x;
            entry(par, 0, b, i, c, x, g);
            lin += a.w[c] * x;
          }
          lin = warp_sum(lin);
        }
        if (lane == 0) sLin = lin;
        sa_bar();
        sa_bar();
        if (a.k1) {
          const T mult = sMult;
          for (uint32_t i = lane; i < nnz; i += 32) {
            uint32_t c, g; T x;
            entry(par, 0, b, i, c, x, g);
            const T gh = mult * x;
            a.gw[c] = gh;
            a.w[c] = sgda_step(a.w[c], gh, lr, T(a.lam_w[g]));
          }
        }
        sa_bar();
      } else {
        if (t + 1 < a.t_end) stage(t + 1);
        sa_bar();
        reduce_mult(nwA, T(rY[par][0]));
        sa_bar();
        if (lane == 0) {
          double s[6] = {sW0, 0, 0, 0, 0, 0};
          double sq = 0.0;
          intercept_step<T, FMWR_SGD, false>(s, (double)sMult, a.k0, sq, a.sp);
          sW0 = s[0];
        }
        sa_bar();
      }
    }
    if (!lam_step) continue;
    // ================= lambda step on the validation row =================
    {
      const uint32_t b = rB[par][1], e = rE[par][1], nnz = e - b;
      const int nwA = (int)((min(nnz, (uint32_t)SLOTS) + SPW - 1) / SPW);
      // group of the validation row's non-zero j: staged, or written by the linear warp before the third barrier below
      auto vgrp = [&](uint32_t j) -> uint32_t { return j < (uint32_t)RN ? (uint32_t)rGrp[par][1][j] : a.cg[j]; };
      if (warp < SA_FW) {
        const bool act = warp < nwA;
        T kth[CH][VN], kla[CH][VN];         // the first round's v and look-ahead v'
        // v' of non-zero i's vector vi from the current v, its last gradient and its group's lambda
        auto lookahead = [&](size_t off, uint32_t g, int vi, T (&th)[VN], T (&la)[VN]) {
          T gh[VN];
          vec_to_arr(reinterpret_cast<const V16*>(a.v + off)[vi], th);
          vec_to_arr(reinterpret_cast<const V16*>(a.gv + off)[vi], gh);
          const double* lv = a.lam_v + (size_t)g * kp + vi * VN;
#pragma unroll
          for (int k = 0; k < VN; ++k) la[k] = sgda_step(th[k], gh[k], lr, T(lv[k]));
        };
        if (act) {
          T S[CH][VN];
          T qsum = T(0);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
#pragma unroll
            for (int k = 0; k < VN; ++k) S[ch][k] = T(0);
          for (uint32_t i0 = 0; i0 < nnz; i0 += SLOTS) {
            const uint32_t i = i0 + slot;
            if (i < nnz) {
              uint32_t c, g; T x;
              entry(par, 1, b, i, c, x, g);
#pragma unroll
              for (int ch = 0; ch < CH; ++ch) {
                T th[VN], la[VN];
                lookahead((size_t)c * kp, g, ch * LPR + l, th, la);
#pragma unroll
                for (int k = 0; k < VN; ++k) {
                  const T tt = la[k] * x;
                  S[ch][k] += tt;
                  qsum += tt * tt;
                  if (i0 == 0) { kth[ch][k] = th[k]; kla[ch][k] = la[k]; }
                }
              }
            }
          }
#pragma unroll
          for (int o = LPR; o < 32; o <<= 1)
#pragma unroll
            for (int ch = 0; ch < CH; ++ch)
#pragma unroll
              for (int k = 0; k < VN; ++k) S[ch][k] += __shfl_xor_sync(0xffffffffu, S[ch][k], o);
          const T part = warp_sum(T(-0.5) * qsum);
          if (lane < LPR) {
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) sS[warp][ch * LPR + l] = arr_to_vec(S[ch]);
          }
          if (lane == 0) sPart[warp] = part;
        }
        sa_bar();
        sa_bar();
        if (act) {
          T Sf[CH][VN];
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) vec_to_arr(sSf[ch * LPR + l], Sf[ch]);
          for (uint32_t i0 = 0; i0 < nnz; i0 += SLOTS) {
            const uint32_t i = i0 + slot;
            if (i < nnz) {
              uint32_t c, g; T x;
              entry(par, 1, b, i, c, x, g);
#pragma unroll
              for (int ch = 0; ch < CH; ++ch) {
                const int vi = ch * LPR + l;
                T th[VN], la[VN];
                if (i0 == 0) {
#pragma unroll
                  for (int k = 0; k < VN; ++k) { th[k] = kth[ch][k]; la[k] = kla[ch][k]; }
                } else {
                  lookahead((size_t)c * kp, g, vi, th, la);
                }
                double* out = a.cv + (size_t)i * kp + vi * VN;
#pragma unroll
                for (int k = 0; k < VN; ++k) out[k] = (double)sgda_v_term(Sf[ch][k], th[k], la[k], x);
              }
            }
          }
        }
        sa_bar();
        if (act) {
          const double mult = (double)sMult;
          // leaders: the first non-zero of each group in the row sums the group's terms in row order and steps its lambda
          for (uint32_t i0 = 0; i0 < nnz; i0 += SLOTS) {
            const uint32_t i = i0 + slot;
            if (i < nnz) {
              const uint32_t g = vgrp(i);
              bool lead = true;
              for (uint32_t j = 0; j < i && lead; ++j) lead = vgrp(j) != g;
              if (lead) {
                double acc[CH][VN];
#pragma unroll
                for (int ch = 0; ch < CH; ++ch)
#pragma unroll
                  for (int k = 0; k < VN; ++k) acc[ch][k] = 0.0;
                for (uint32_t j = i; j < nnz; ++j) {
                  if (vgrp(j) != g) continue;
#pragma unroll
                  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
                    for (int k = 0; k < VN; ++k) acc[ch][k] += a.cv[(size_t)j * kp + (ch * LPR + l) * VN + k];
                }
#pragma unroll
                for (int ch = 0; ch < CH; ++ch) {
                  double* lv = a.lam_v + (size_t)g * kp + (ch * LPR + l) * VN;
#pragma unroll
                  for (int k = 0; k < VN; ++k) lv[k] = sgda_lambda_step(lv[k], a.lr, mult, acc[ch][k]);
                }
              }
            }
          }
        }
        sa_bar();
      } else if (warp == W_LIN) {
        T lin = T(0);
        for (uint32_t i = lane; i < nnz; i += 32) {
          uint32_t c, g; T x;
          entry(par, 1, b, i, c, x, g);
          if (i >= (uint32_t)RN) a.cg[i] = g;
          if (a.k1) {
            const T th = a.w[c];
            lin += sgda_step(th, a.gw[c], lr, T(a.lam_w[g])) * x;
            a.cw[i] = (double)(x * th);
          }
        }
        if (a.k1) lin = warp_sum(lin);
        if (lane == 0) sLin = lin;
        sa_bar();
        sa_bar();
        sa_bar();
        if (a.k1) {
          const double mult = (double)sMult;
          for (uint32_t i = lane; i < nnz; i += 32) {
            const uint32_t g = vgrp(i);
            bool lead = true;
            for (uint32_t j = 0; j < i && lead; ++j) lead = vgrp(j) != g;
            if (!lead) continue;
            double acc = 0.0;
            for (uint32_t j = i; j < nnz; ++j)
              if (vgrp(j) == g) acc += a.cw[j];
            a.lam_w[g] = sgda_lambda_step(a.lam_w[g], a.lr, mult, acc);
          }
        }
        sa_bar();
      } else {
        sa_bar();
        reduce_mult(nwA, T(rY[par][1]));
        sa_bar();
        sa_bar();
        sa_bar();
      }
    }
  }
  if (tid == W_PIPE * 32) a.scal[0] = sW0;
}

template <class T>
struct SgdaLaunch {
  fmwr_ctx* ctx; SgdaArgs<T> args;
  template <class TT, int LPR, int CH>
  void run() { FMWR_LAUNCH(ctx, (sgda_kernel<TT, LPR, CH>), 1, SA_THREADS, 0, args); }
};

template <class T>
static void train_sgda_t(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, fmwr_data* valid,
                         double* lambda_w, double* lambda_v)
{
  cudaStream_t st = ctx->stream;
  const int64_t p = m->p;
  const int kp = m->kp, k = m->k;
  const int G = s->attr_group ? s->n_groups : 1;
  const int skip_row0 = (s->compat & FMWR_COMPAT_SKIP_ROW0) ? 1 : 0;
  std::vector<uint32_t> order_host = visit_order_host(d, s);
  model_alloc_state(m, 0, 0, false);         // the gradients below are call-owned: the handle keeps no optimizer state
  if (order_host.empty() && d->n <= skip_row0) return;   // no row to visit

  SgdaArgs<T> a;
  memset(&a, 0, sizeof a);
  a.rowptr = d->rowptr.p; a.col = d->col.p; a.val = d->val.p; a.y = d->y.p;
  a.vrowptr = valid->rowptr.p; a.vcol = valid->col.p; a.vval = valid->val.p; a.vy = valid->y.p;
  a.w = (T*)m->w.p; a.v = (T*)m->v.p; a.scal = (double*)m->scal.p;
  a.kp = kp; a.k0 = m->cfg.keep_w0; a.k1 = m->cfg.keep_w1; a.task = m->cfg.task;
  a.n_val = valid->n;
  a.skip_row0 = skip_row0;
  a.sp = make_params<T>(m, s);
  a.lo = s->min_target; a.hi = s->max_target;
  a.lr = s->learn_rate;

  DBuf<uint32_t> order_dev;
  if (!order_host.empty()) {
    order_dev.alloc(order_host.size());
    FMWR_CUDA(cudaMemcpyAsync(order_dev.p, order_host.data(), 4 * order_host.size(), cudaMemcpyHostToDevice, st));
    a.order = order_dev.p;
  }
  a.period = a.order ? (int64_t)order_host.size() : d->n - skip_row0;
  // T0: an explicit visit_order is one pass; the random_step sequence is its sweeps cut at max_iter, each sweep strictly
  // ascending, so its first pass ends where the row index first fails to increase (all of it when max_iter ends the first sweep)
  a.t0 = a.period;
  if (a.order && !(s->visit_order && s->n_visit > 0))
    for (int64_t i = 1; i < a.period; ++i)
      if (order_host[i] <= order_host[i - 1]) { a.t0 = i; break; }

  // groups (u16), lambdas (padded to kp, zeros past k), gradients
  std::vector<uint16_t> grp_host(p, 0);
  if (s->attr_group)
    for (int64_t i = 0; i < p; ++i) grp_host[i] = (uint16_t)s->attr_group[i];
  std::vector<double> lv_host((size_t)G * kp, 0.0);
  for (int g = 0; g < G; ++g)
    for (int f = 0; f < k; ++f) lv_host[(size_t)g * kp + f] = lambda_v[(size_t)g * k + f];
  DBuf<uint16_t> grp; DBuf<double> lam_w, lam_v; DBuf<char> gw, gv;
  grp.alloc(p); lam_w.alloc(G); lam_v.alloc((size_t)G * kp);
  gw.alloc((size_t)p * sizeof(T)); gv.alloc((size_t)p * kp * sizeof(T));
  FMWR_CUDA(cudaMemcpyAsync(grp.p, grp_host.data(), 2 * p, cudaMemcpyHostToDevice, st));
  FMWR_CUDA(cudaMemcpyAsync(lam_w.p, lambda_w, 8 * G, cudaMemcpyHostToDevice, st));
  FMWR_CUDA(cudaMemcpyAsync(lam_v.p, lv_host.data(), 8 * lv_host.size(), cudaMemcpyHostToDevice, st));
  gw.zero(st); gv.zero(st);
  a.grp = grp.p; a.lam_w = lam_w.p; a.lam_v = lam_v.p; a.gw = (T*)gw.p; a.gv = (T*)gv.p;

  // scratch of the validation row's terms, sized by its longest row
  std::vector<uint32_t> vptr(valid->n + 1);
  FMWR_CUDA(cudaMemcpyAsync(vptr.data(), valid->rowptr.p, 4 * vptr.size(), cudaMemcpyDeviceToHost, st));
  FMWR_CUDA(cudaStreamSynchronize(st));
  uint32_t max_nnz = 1;
  for (int64_t i = 0; i < valid->n; ++i) max_nnz = std::max(max_nnz, vptr[i + 1] - vptr[i]);
  DBuf<double> cv, cw; DBuf<uint32_t> cg;
  cv.alloc((size_t)max_nnz * kp); cw.alloc(max_nnz); cg.alloc(max_nnz);
  a.cv = cv.p; a.cw = cw.p; a.cg = cg.p;

  Tracker trk(ctx, m, s, tr, nullptr);
  const int step = trk.step;
  const int64_t max_iter = s->max_iter;
  int64_t iter = 0;
  while (iter < max_iter) {
    // launches end at the tracker's records (after samples 0, step, 2 step, ... and max_iter-1), as train_exact_t's do
    const int64_t next = step > 0 ? std::min<int64_t>((iter + step - 1) / step * step + 1, max_iter) : max_iter;
    a.t_begin = iter; a.t_end = next;
    SgdaLaunch<T> L{ctx, a};
    dispatch_layout<T>(kp, L);
    iter = next;
    if (trk.due(iter - 1) && trk.record(iter - 1, tracker_score(ctx, m, d, s))) break;
  }
  trk.restore_best();
  std::vector<double> lv_out((size_t)G * kp);
  FMWR_CUDA(cudaMemcpyAsync(lambda_w, lam_w.p, 8 * G, cudaMemcpyDeviceToHost, st));
  FMWR_CUDA(cudaMemcpyAsync(lv_out.data(), lam_v.p, 8 * lv_out.size(), cudaMemcpyDeviceToHost, st));
  FMWR_CUDA(cudaStreamSynchronize(st));
  for (int g = 0; g < G; ++g)
    for (int f = 0; f < k; ++f) lambda_v[(size_t)g * k + f] = lv_out[(size_t)g * kp + f];
  trk.write_trace(iter);
}

void train_sgda(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, fmwr_data* valid,
                double* lambda_w, double* lambda_v)
{
  if (m->prec == FMWR_F64) train_sgda_t<double>(ctx, m, d, s, tr, valid, lambda_w, lambda_v);
  else train_sgda_t<float>(ctx, m, d, s, tr, valid, lambda_w, lambda_v);
}

}  // namespace fmwr
