// What one SGD / FTRL-Proximal / TDAP step does to a coordinate, its optimizer state and the intercept, shared by the
// exact (batch = 1) and minibatch kernels.  The kernels only decide where operands come from and where results go.
//
// Every step takes the coordinate's gradient g (for the exact mode g is one sample's
// gradient, for the minibatch mode the sum over the batch rows that touch the coordinate),
// the current parameter value and its optimizer state, and returns the new value.
//   SGD   reference src/solver/SGD_Learner.h:106-138 (+ apply_penalty :195-204)
//   FTRL  reference src/solver/FTRL_Learner.h:80-113 (state) and :177-199 (closed-form refresh)
//   TDAP  reference src/solver/TDAP_Learner.h:96-143 (state) and :203-231 (refresh)
#pragma once
#include "common.cuh"

#include <cmath>

namespace fmwr {

template <class T>
struct SolverParams {
  int solver;        // FMWR_SGD / FMWR_FTRL / FMWR_TDAP
  int l1;            // SGD: cumulative-penalty L1 active
  T lr;              // SGD
  T reg_w, reg_v;    // SGD: L2 rate (or L1 rate when l1)
  T reg_w0;          // SGD: L2.w0
  T alpha_w, alpha_v, beta_w, beta_v;   // FTRL / TDAP
  T l1_w, l1_v, l2_w, l2_v;             // FTRL / TDAP refresh
  T egamma;          // TDAP exp(-gamma)
};

// State arrays per coordinate, in this order: SGD q (cumulative L1 only); FTRL z, n; TDAP u, nu, delta, h
constexpr int solver_nst(int solver) { return solver == FMWR_SGD ? 1 : (solver == FMWR_FTRL ? 2 : 4); }

// state arrays the model keeps (SGD without L1 keeps none)
inline int solver_state_count(const SolverParams<double>& sp) { return sp.solver == FMWR_SGD ? sp.l1 : solver_nst(sp.solver); }

template <class T>
SolverParams<T> make_params(const fmwr_model* m, const fmwr_solver_cfg* s)
{
  SolverParams<T> sp;
  memset(&sp, 0, sizeof sp);
  sp.solver = s->solver;
  const fmwr_model_cfg& c = m->cfg;
  if (s->solver == FMWR_SGD) {
    // SGD_Learner::init (reference src/solver/SGD_Learner.h:44-59): any L1 > 0 selects the L1 rates;
    // L1 proper is only used for classification, in regression the L1 rates act as L2 rates.
    double regw, regv; int l1 = 0;
    if (c.l1_w1 > 0 || c.l1_v > 0) { l1 = 1; regw = c.l1_w1; regv = c.l1_v; }
    else { regw = c.l2_w1; regv = c.l2_v; }
    if (c.task != FMWR_CLASSIFICATION) l1 = 0;
    sp.l1 = l1; sp.lr = T(s->learn_rate); sp.reg_w = T(regw); sp.reg_v = T(regv); sp.reg_w0 = T(c.l2_w0);
  } else {
    sp.alpha_w = T(s->alpha_w); sp.alpha_v = T(s->alpha_v); sp.beta_w = T(s->beta_w); sp.beta_v = T(s->beta_v);
    sp.l1_w = T(c.l1_w1); sp.l1_v = T(c.l1_v); sp.l2_w = T(c.l2_w1); sp.l2_v = T(c.l2_v);
    sp.egamma = T(std::exp(-s->gamma));
  }
  return sp;
}

// d/dv_f of the pairwise term for one non-zero: S_f x - v x^2, with the reference's operation order and
// NO fused multiply-add (reference src/solver/SGD_Learner.h:129: `sum * x - v * x * x`).  On a row whose
// only non-zero is this feature S_f == v*x, so the expression is exactly 0 in the reference; a contracted
// FMA would leave a rounding residue of random sign, and TDAP (no beta in its denominator) turns the sign of
// an infinitesimal gradient into a +-alpha jump of the parameter.
__device__ __forceinline__ float fm_grad(float S, float v, float x) { return __fsub_rn(__fmul_rn(S, x), __fmul_rn(__fmul_rn(v, x), x)); }
__device__ __forceinline__ double fm_grad(double S, double v, double x) { return __dsub_rn(__dmul_rn(S, x), __dmul_rn(__dmul_rn(v, x), x)); }

// cumulative-penalty clip (Tsuruoka et al.), reference src/solver/SGD_Learner.h:195-204
template <class T>
__device__ __forceinline__ void sgd_apply_penalty(T& theta, T u, T& q)
{
  // both clips computed, one selected: the same values as the reference's if / else-if, without a divergent branch per element
  const T old = theta;
  const T pos = fmax(T(0), old - (u + q)), neg = fmin(T(0), old + (u - q));
  theta = old > T(0) ? pos : (old < T(0) ? neg : old);
  q += theta - old;
}

// SGD step for one coordinate.  g excludes the learning rate.  q is touched only when l1.
template <class T>
__device__ __forceinline__ T sgd_step(T theta, T g, T lr, T reg, int l1, T u, T& q)
{
  theta -= lr * g;
  if (l1) sgd_apply_penalty(theta, u, q);
  else theta -= lr * reg * theta;
  return theta;
}

// Throughput-mode arithmetic: MUFU approximations (sqrt.approx / rcp.approx, <= 2 ulp) instead of the IEEE
// sequences (~10 instructions each, and each ends a basic block) -- the minibatch update kernel is issue-bound on
// them and the exact (batch = 1) kernel serialises a vector's elements behind them.  FAST is only ever set for
// fp32 FTRL / TDAP kernels; SGD has no sqrt / div, and every fp64 instantiation keeps IEEE operations.
template <bool FAST> __device__ __forceinline__ float m_sqrt(float x)
{
  if (FAST) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
  return sqrtf(x);
}
template <bool FAST> __device__ __forceinline__ double m_sqrt(double x) { return sqrt(x); }
template <bool FAST> __device__ __forceinline__ float m_div(float a, float b) { return FAST ? __fdividef(a, b) : a / b; }
template <bool FAST> __device__ __forceinline__ double m_div(double a, double b) { return a / b; }

// FTRL-Proximal: state (z, n) in/out, returns refreshed theta
// SEL: compute the closed form unconditionally and select (same value; no branch, so the elements of a vector
// interleave in the latency-bound exact kernel)
template <class T, bool FAST = false, bool SEL = false>
__device__ __forceinline__ T ftrl_step(T theta, T g, T& z, T& n, T alpha, T beta, T l1, T l2)
{
  const T n_old = n;
  n = n_old + g * g;
  const T sq = m_sqrt<FAST>(n);
  const T sigma = m_div<FAST>(sq - m_sqrt<FAST>(n_old), alpha);
  z += g - sigma * theta;
  if (!SEL && fabs(z) <= l1) return T(0);
  const T sign = z < T(0) ? T(-1) : T(1);
  const T r = -m_div<FAST>(z - sign * l1, m_div<FAST>(beta + sq, alpha) + l2);
  return (SEL && fabs(z) <= l1) ? T(0) : r;
}

// TDAP state update: (u, nu, delta, h) in/out; returns z = nu - h
template <class T, bool FAST = false>
__device__ __forceinline__ T tdap_state(T theta, T g, T& u, T& nu, T& delta, T& h, T alpha, T egamma)
{
  const T u_old = u;
  u = u_old + g * g;
  nu += g;
  const T sigma = m_div<FAST>(m_sqrt<FAST>(u) - m_sqrt<FAST>(u_old), alpha);
  delta = egamma * (delta + sigma);
  h = egamma * (h + sigma * theta);
  return nu - h;
}

template <class T, bool FAST = false, bool SEL = false>
__device__ __forceinline__ T tdap_refresh(T z, T delta, T l1, T l2)
{
  if (!SEL && fabs(z) <= l1) return T(0);
  const T sign = z < T(0) ? T(-1) : T(1);
  const T r = -m_div<FAST>(z - sign * l1, delta + l2);
  return (SEL && fabs(z) <= l1) ? T(0) : r;
}

// One step of a coordinate: th (in/out), its gradient g, its state st (in/out, solver_nst(SOLVER) values in the order above).
// LIN: the linear-weight hyper-parameters, else the factors'.  l1: SGD's cumulative L1 is on (st[0] = q; u = its total after
// this step), a constant in the minibatch kernels and a run-time flag in the exact ones.  SEL: see ftrl_step.
template <class T, int SOLVER, bool LIN, bool FAST, bool SEL>
__device__ __forceinline__ T coord_step(T th, T g, T (&st)[solver_nst(SOLVER)], const SolverParams<T>& sp, int l1, T u)
{
  if constexpr (SOLVER == FMWR_SGD) {
    T q = l1 ? st[0] : T(0);
    th = sgd_step(th, g, sp.lr, LIN ? sp.reg_w : sp.reg_v, l1, u, q);
    st[0] = q;
    return th;
  } else if constexpr (SOLVER == FMWR_FTRL) {
    return ftrl_step<T, FAST, SEL>(th, g, st[0], st[1], LIN ? sp.alpha_w : sp.alpha_v, LIN ? sp.beta_w : sp.beta_v,
                                   LIN ? sp.l1_w : sp.l1_v, LIN ? sp.l2_w : sp.l2_v);
  } else {
    const T z = tdap_state<T, FAST>(th, g, st[0], st[1], st[2], st[3], LIN ? sp.alpha_w : sp.alpha_v, sp.egamma);
    return tdap_refresh<T, FAST, SEL>(z, st[2], LIN ? sp.l1_w : sp.l1_v, LIN ? sp.l2_w : sp.l2_v);
  }
}

// The same step on the VN elements of one 16-byte vector of a factor row.
template <class T, int SOLVER, bool LIN, bool FAST, bool SEL, int VN>
__device__ __forceinline__ void coord_step(T (&th)[VN], const T (&g)[VN], T (&st)[solver_nst(SOLVER)][VN], const SolverParams<T>& sp, int l1, T u)
{
  constexpr int NS = solver_nst(SOLVER);
#pragma unroll
  for (int i = 0; i < VN; ++i) {
    T s[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) s[k] = st[k][i];
    th[i] = coord_step<T, SOLVER, LIN, FAST, SEL>(th[i], g[i], s, sp, l1, u);
#pragma unroll
    for (int k = 0; k < NS; ++k) st[k][i] = s[k];
  }
}

// Gradient of a minibatch segment (one feature's rows in one batch): Gw for the linear weight, Gv[CH][VN] for the lane's
// factor vectors th.  seg_grad_entry adds one entry (the row's multiplier m, the value x, the row's S-cache vectors s;
// FIRST: the segment's first entry, which sets the sums); seg_grad_close ends the segment.
// TDAP keeps the per-entry gradient form of the exact mode (see fm_grad: a rounding residue flips theta by +-alpha);
// SGD / FTRL sum  A_f = sum_r (m_r x_r) S_rf  and  b = sum_r m_r x_r^2  and form  G_f = A_f - v_f b  once (the same
// value up to rounding; at batch = 1 it differs from the exact mode's per-entry form by an ulp, not by a step)
template <int SOLVER, bool FIRST = false, class T, int CH, int VN>
__device__ __forceinline__ void seg_grad_entry(T& Gw, T& bsum, T (&Gv)[CH][VN], const T (&th)[CH][VN], T m, T x,
                                               const typename Vec<T>::type (&s)[CH])
{
  constexpr bool ENTRY_FORM = SOLVER == FMWR_TDAP;
  const T mx = m * x;
  if (FIRST) { Gw = mx; bsum = mx * x; }
  else {
    Gw += mx;
    if (!ENTRY_FORM) bsum += mx * x;
  }
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    T sa[VN];
    vec_to_arr(s[ch], sa);
#pragma unroll
    for (int k = 0; k < VN; ++k) {
      const T t = ENTRY_FORM ? m * fm_grad(sa[k], th[ch][k], x) : mx * sa[k];
      Gv[ch][k] = FIRST ? t : Gv[ch][k] + t;
    }
  }
}

template <int SOLVER, class T, int CH, int VN>
__device__ __forceinline__ void seg_grad_close(T (&Gv)[CH][VN], const T (&th)[CH][VN], T bsum)
{
  if constexpr (SOLVER != FMWR_TDAP) {
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int k = 0; k < VN; ++k) Gv[ch][k] = Gv[ch][k] - th[ch][k] * bsum;
  }
}

// One step of the intercept w0 (fp64 as the reference's doubles) on s = {w0, state}: FTRL s[1] z, s[2] n; TDAP s[1] u,
// s[2] nu, s[3] delta, s[4] h, s[5] z.  g: its gradient (SGD: the caller's batch mean).  sq: the square root of the
// accumulator (FTRL s[2], TDAP s[1]) before the step in, after it out -- carried by the exact kernels between samples so
// that their serial chain takes one sqrt per step.  INV: multiply by inv_alpha_w instead of dividing by alpha_w (fp32
// exact kernels: a 1-ulp fp64 change, nine digits below the fp32 parameters, off the serial chain's longest operation).
//   SGD_Learner.h:106-109, FTRL_Learner.h:80-86 and :161, TDAP_Learner.h:96-105 and :192
template <class T, int SOLVER, bool INV>
__device__ __forceinline__ void intercept_step(double (&s)[6], double g, int k0, double& sq, const SolverParams<T>& sp,
                                               double inv_alpha_w = 0.0)
{
  if (SOLVER == FMWR_SGD) {
    if (k0) s[0] -= (double)sp.lr * (g + (double)sp.reg_w0 * s[0]);
  } else if (SOLVER == FMWR_FTRL) {
    if (k0) {
      s[2] += g * g;
      const double sq1 = sqrt(s[2]);
      const double delta = INV ? (sq1 - sq) * inv_alpha_w : (sq1 - sq) / (double)sp.alpha_w;
      sq = sq1;
      s[1] += g - delta * s[0];
    }
    s[0] = -s[1] * (double)sp.alpha_w / ((double)sp.beta_w + sq);     // unconditional
  } else {
    if (k0) {
      s[1] += g * g; s[2] += g;
      const double sq1 = sqrt(s[1]);
      const double sigma = INV ? (sq1 - sq) * inv_alpha_w : (sq1 - sq) / (double)sp.alpha_w;
      sq = sq1;
      s[3] = (double)sp.egamma * (s[3] + sigma);
      s[4] = (double)sp.egamma * (s[4] + sigma * s[0]);
      s[5] = s[2] - s[4];
    }
    s[0] = -s[5] / s[3];                                                 // 0/0 = NaN when keep.w0 is false
  }
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

}  // namespace fmwr
