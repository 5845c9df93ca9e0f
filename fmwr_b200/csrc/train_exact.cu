// Exact (batch = 1) SGD / FTRL-Proximal / TDAP in the reference's visit order.
//
// Replaces SGD_Learner::learn, FTRL_Learner::learn + calculate_param, TDAP_Learner::learn +
// calculate_param (reference src/solver/SGD_Learner.h:79-178, FTRL_Learner.h:64-202,
// TDAP_Learner.h:79-233).  Samples are strictly serial (w0 is read by every forward and written
// by every update), so the parallelism is INSIDE a sample: one persistent CTA walks the visit
// sequence.  Within one sample every coordinate update is independent given `mult` and the
// frozen S_f (each (f, j) is touched once), which is exactly what the reference's f-outer /
// nnz-inner loops compute.
//
// The sample time is a chain of latencies (DRAM ~1000 cycles, shared memory ~30, IEEE div/sqrt
// sequences that end basic blocks), measured with clock64() per role (profiles/r01_summary.md).
// The CTA is therefore warp-specialised, and each role runs only its own short program:
//   * factor warps (0 .. FW-1): thread (slot, l) owns non-zero `slot` of the row and the 16-byte
//     vector l of that feature's factor row; warps without a non-zero only hit the barriers;
//   * the linear warp: lane = non-zero (two per lane in registers), owns w_j and its state;
//   * the pipeline warp: runs ahead of the sample being processed -- visit index (t+4), row bounds
//     and label (t+3), the row's first column/value entries (t+2) into shared-memory rings,
//     and an L2 prefetch of every parameter / state line sample t+1 will touch -- and owns w0 and
//     the scalar optimizer state (fp64, double-buffered by sample parity so it is updated while
//     the other warps still read it).  The CSR arrays are read-only and L2 is the coherence point,
//     so running ahead cannot observe stale data.
// Rows that fit one round (nnz <= SLOTS) read theta and its state once, with the forward gather,
// and keep them in registers for the update.  Three barriers per sample: partials ready, S_f and the
// multiplier published (summed by the pipeline warp alone), updates done.
// fp32 models use the branch-free MUFU exp/sqrt/rcp forms (<= 2 ulp, the same order as fp32 rounding
// itself; lets the four elements of a vector interleave); fp64 keeps IEEE operations throughout.
#include "forward.cuh"
#include "coord.cuh"

#include <cmath>
#include <cstdlib>

namespace fmwr {

constexpr int EX_THREADS = 512;
constexpr int EX_WARPS = EX_THREADS / 32;
constexpr int EX_FW = EX_WARPS - 2;          // factor warps
constexpr int EX_NL = 2;                     // non-zeros per lane the linear warp keeps in registers

template <class T>
struct ExactArgs {
  const uint32_t* rowptr; const uint32_t* col; const float* val; const float* y;
  T* w; T* v; double* scal;
  T* sw[4]; T* sv[4];
  int kp, k0, k1, task;
  int64_t n;
  const uint32_t* order;     // explicit visit order (NULL: scan)
  int64_t order_len;
  int skip_row0;             // F5: scan rows 1..n-1
  int64_t t_begin, t_end;    // sample counters of this launch
  int tdap_zw_index;         // F6
  int nohazard;              // tests only (FMWR_EXACT_NOHAZARD=1): the pipeline does not wait for column hazards
  SolverParams<T> sp;
  double lo, hi;
};

// CTA barrier reached from role-specific code (every warp arrives whole, the same number of times per sample)
__device__ __forceinline__ void ex_bar() { asm volatile("bar.sync 0;" ::: "memory"); }

template <class T, int LPR, int CH, int SOLVER>
__global__ void __launch_bounds__(EX_THREADS, 1) exact_kernel(ExactArgs<T> a)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int SLOTS = EX_FW * 32 / LPR;
  constexpr int SPW = 32 / LPR;             // slots per factor warp
  constexpr int NS = solver_nst(SOLVER);   // state arrays (SGD: only with L1)
  constexpr bool KEEP = (CH == 1);          // registers for theta + state only at one vector per lane
  constexpr bool FAST = sizeof(T) == 4;     // fp32: MUFU exp / sqrt / rcp (SGD only has the multiplier's exp and rcp)
  constexpr int RING = 8, CRING = 4;
  constexpr int RN = SLOTS > 32 * EX_NL ? SLOTS : 32 * EX_NL;   // non-zeros of a row staged in the shared-memory ring
  constexpr int NC = (RN + 31) / 32;        // ring entries per pipeline lane
  constexpr int NL = EX_NL;
  constexpr int W_PIPE = EX_FW, W_LIN = EX_FW + 1;
  constexpr int LINE = 128 / (int)sizeof(T);
  __shared__ V16 sS[EX_FW][LPR * CH];
  __shared__ T sPart[EX_FW];
  __shared__ T sLin;
  __shared__ V16 sSf[LPR * CH];             // S_f of the sample, summed over the factor warps by the pipeline warp
  __shared__ T sMult;
  __shared__ double sc[2][8];               // w0 and the scalar optimizer state, by sample parity
  __shared__ uint32_t rRow[RING], rB[RING], rE[RING];
  __shared__ float rY[RING];
  __shared__ uint32_t rCol[CRING][RN];
  __shared__ float rVal[CRING][RN];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = tid / LPR, l = tid % LPR;          // factor warps only
  const int kp = a.kp;
  const SolverParams<T> sp = a.sp;
  const bool sgd_l1 = (SOLVER == FMWR_SGD) && sp.l1;
  const bool has_state = (SOLVER != FMWR_SGD) || sp.l1;
  if (a.t_begin >= a.t_end) return;
  if (tid < 8) sc[a.t_begin & 1][tid] = a.scal[tid];

  // ---- pipeline prologue: rings for the first samples
  const int64_t period = a.order ? a.order_len : (a.skip_row0 ? a.n - 1 : a.n);
  int64_t pos = 0;                          // visit cursor (pipeline warp, lane 0)
  auto row_at = [&](int64_t q) -> uint32_t { return a.order ? a.order[q] : (uint32_t)(a.skip_row0 ? q + 1 : q); };
  if (tid == W_PIPE * 32) {
    pos = a.t_begin % period;
    for (int i = 0; i < 4 && a.t_begin + i < a.t_end; ++i) {
      rRow[(a.t_begin + i) & (RING - 1)] = row_at(pos);
      if (++pos == period) pos = 0;
    }
  }
  __syncthreads();
  if (tid < 3 && a.t_begin + tid < a.t_end) {
    const int s = (int)((a.t_begin + tid) & (RING - 1));
    const uint32_t r = rRow[s];
    rB[s] = a.rowptr[r]; rE[s] = a.rowptr[r + 1]; rY[s] = a.y[r];
  }
  __syncthreads();
  for (int i = 0; i < 2; ++i) {
    const int64_t s = a.t_begin + i;
    if (s < a.t_end && tid < RN) {
      const uint32_t j = rB[s & (RING - 1)] + tid;
      if (j < rE[s & (RING - 1)]) { rCol[s & (CRING - 1)][tid] = a.col[j]; rVal[s & (CRING - 1)][tid] = a.val[j]; }
    }
  }
  __syncthreads();
  // sqrt of the w0 accumulator (FTRL n, TDAP u) is carried between samples by its owner
  double sq_acc = 0.0;
  // fp32 models: the w0 state stays fp64 but its one constant divisor becomes a multiplication (intercept_step); fp64 models
  // keep the reference's division
  const double inv_alpha_w = 1.0 / (double)sp.alpha_w;
  if (tid == W_PIPE * 32) sq_acc = sqrt(SOLVER == FMWR_FTRL ? sc[a.t_begin & 1][2] : sc[a.t_begin & 1][1]);

#ifdef FMWR_EXACT_PROF
  // per-role timeline (cycles per sample); a barrier's wait shows up in the section AFTER it (deferred blocking)
  long long pt[4] = {0, 0, 0, 0};
#define PROF(i) { const long long c_ = clock64(); pt[i] += c_ - p0; p0 = c_; }
#else
#define PROF(i)
#endif
  for (int64_t t = a.t_begin; t < a.t_end; ++t) {
#ifdef FMWR_EXACT_PROF
    long long p0 = clock64();
#endif
    double* const scur = sc[t & 1];
    double* const snext = sc[(t + 1) & 1];
    const uint32_t b = rB[t & (RING - 1)], e = rE[t & (RING - 1)];
    const uint32_t nnz = e - b;
    const T yv = T(rY[t & (RING - 1)]);
    const uint32_t* const ccol = rCol[t & (CRING - 1)];
    const float* const cval = rVal[t & (CRING - 1)];
    const uint32_t used = min(nnz, (uint32_t)SLOTS);
    const int nwA = (int)((used + SPW - 1) / SPW);      // factor warps holding entries

    // pipeline warp, between the two mid-sample barriers: S_f over the factor warps (lane = factor), the score
    // and the multiplier, published through shared memory -- one warp's ~60 instructions instead of every warp's
    auto reduce_mult = [&]() -> T {
      T acc = T(0);
      T* const sf_out = reinterpret_cast<T*>(sSf);
      for (int f = lane; f < LPR * CH * VN; f += 32) {
        T sf = T(0);
#pragma unroll
        for (int w2 = 0; w2 < EX_FW; ++w2)
          if (w2 < nwA) sf += reinterpret_cast<const T*>(sS[w2])[f];
        sf_out[f] = sf;
        acc += T(0.5) * sf * sf;
      }
      if (lane < nwA) acc += sPart[lane];
      acc = warp_sum(acc);
      acc += sLin;
      const T score = (a.k0 ? T(scur[0]) : T(0)) + acc;          // Model::predict, reference src/core/Model.h:75-103
      // calculate_grad_mult
      const T mult = FAST ? grad_mult_fast(a.task, score, yv, T(a.lo), T(a.hi)) : grad_mult<T>(a.task, score, yv, T(a.lo), T(a.hi));
      if (lane == 0) sMult = mult;
      return mult;
    };

    if (warp < EX_FW) {
      // =========================== factor warps ===========================
      const bool act = warp < nwA;
      const bool single = KEEP && nnz <= (uint32_t)SLOTS;
      T kth[VN], kst[NS][VN];
      uint32_t c0 = 0; T x0 = T(0);
      if (act) {
        T S[CH][VN];
        T qsum = T(0);
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
#pragma unroll
          for (int i = 0; i < VN; ++i) S[ch][i] = T(0);
        for (uint32_t j0 = b; j0 < e; j0 += SLOTS) {
          const uint32_t j = j0 + slot;
          if (j < e) {
            uint32_t c; T x;
            if (j0 == b) { c = ccol[slot]; x = T(cval[slot]); c0 = c; x0 = x; }
            else { c = a.col[j]; x = T(a.val[j]); }
            const size_t off = (size_t)c * kp;
            const V16* vr = reinterpret_cast<const V16*>(a.v + off);
            if (single && has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) vec_to_arr(reinterpret_cast<const V16*>(a.sv[s] + off)[l], kst[s]);
            }
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) {
              T arr[VN];
              vec_to_arr(vr[ch * LPR + l], arr);
#pragma unroll
              for (int i = 0; i < VN; ++i) {
                const T tt = arr[i] * x;
                S[ch][i] += tt;
                qsum += tt * tt;
                if (KEEP) kth[i] = arr[i];
              }
            }
          }
        }
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1)
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
#pragma unroll
            for (int i = 0; i < VN; ++i) S[ch][i] += __shfl_xor_sync(0xffffffffu, S[ch][i], o);
        PROF(0)
        const T part = warp_sum(T(-0.5) * qsum);
        if (lane < LPR) {
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) sS[warp][ch * LPR + l] = arr_to_vec(S[ch]);
        }
        if (lane == 0) sPart[warp] = part;
      }
      PROF(1)
      ex_bar();
      ex_bar();
      if (act) {
        const T mult = sMult;
        PROF(2)
        T Sf[CH][VN];
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) vec_to_arr(sSf[ch * LPR + l], Sf[ch]);
        const T u_v = sgd_l1 ? T(scur[2]) : T(0);
        for (uint32_t j0 = b; j0 < e; j0 += SLOTS) {
          const uint32_t j = j0 + slot;
          if (j < e) {
            uint32_t c; T x;
            if (j0 == b) { c = c0; x = x0; } else { c = a.col[j]; x = T(a.val[j]); }
            const size_t off = (size_t)c * kp;
            V16* vr = reinterpret_cast<V16*>(a.v + off);
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) {
              const int vi = ch * LPR + l;
              T th[VN], st[NS][VN] = {};
              if (single) {
#pragma unroll
                for (int i = 0; i < VN; ++i) th[i] = kth[i];
                if (has_state) {
#pragma unroll
                  for (int s = 0; s < NS; ++s)
#pragma unroll
                    for (int i = 0; i < VN; ++i) st[s][i] = kst[s][i];
                }
              } else {
                vec_to_arr(vr[vi], th);
                if (has_state) {
#pragma unroll
                  for (int s = 0; s < NS; ++s) vec_to_arr(reinterpret_cast<const V16*>(a.sv[s] + off)[vi], st[s]);
                }
              }
              // element by element, each gradient formed just before its step: the fp64 steps branch, and gradients formed ahead
              // would stay live across those branches (registers)
#pragma unroll
              for (int i = 0; i < VN; ++i) {
                T s[NS];
                for (int k = 0; k < NS; ++k) s[k] = st[k][i];
                th[i] = coord_step<T, SOLVER, false, FAST, FAST>(th[i], mult * fm_grad(Sf[ch][i], th[i], x), s, sp, sp.l1, u_v);
                for (int k = 0; k < NS; ++k) st[k][i] = s[k];
              }
              if (has_state) {
#pragma unroll
                for (int s = 0; s < NS; ++s) reinterpret_cast<V16*>(a.sv[s] + off)[vi] = arr_to_vec(st[s]);
              }
              vr[vi] = arr_to_vec(th);
            }
          }
        }
      }
      PROF(3)
      ex_bar();
    } else if (warp == W_LIN) {
      // =========================== linear warp: lane = non-zero ===========================
      const bool lsingle = nnz <= 32u * NL;      // all of the row's w_j (and state) stay in registers
      uint32_t kc[NL]; T kx[NL], kw[NL], ksw[NL][NS];
      T lin = T(0);
      auto entry = [&](uint32_t i, uint32_t& c, T& x) {
        if (i < (uint32_t)RN) { c = ccol[i]; x = T(cval[i]); } else { c = a.col[b + i]; x = T(a.val[b + i]); }
      };
      if (a.k1) {
        if (lsingle) {
          // branch-free on purpose: all shared-memory reads, then all global reads.  With a branch per non-zero the
          // second non-zero's address arithmetic waited on the scoreboard of the first one's loads (ncu source page:
          // two serialised DRAM round trips); lanes past the row's end read element 0 and are masked by x = 0.
#pragma unroll
          for (int q = 0; q < NL; ++q) {
            const uint32_t i = q * 32 + lane;            // < 32 * NL <= RN
            const bool ok = i < nnz;
            const uint32_t c = ccol[i];
            const T x = T(cval[i]);
            kc[q] = ok ? c : 0u; kx[q] = ok ? x : T(0);
#pragma unroll
            for (int s = 0; s < NS; ++s) ksw[q][s] = T(0);
          }
#pragma unroll
          for (int q = 0; q < NL; ++q) {
            kw[q] = a.w[kc[q]];
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) ksw[q][s] = a.sw[s][kc[q]];
            }
          }
#pragma unroll
          for (int q = 0; q < NL; ++q) lin += kw[q] * kx[q];
        } else {
          for (uint32_t i = lane; i < nnz; i += 32) {
            uint32_t c; T x;
            entry(i, c, x);
            lin += a.w[c] * x;
          }
        }
        lin = warp_sum(lin);
      }
      if (lane == 0) sLin = lin;
      PROF(1)
      ex_bar();
      ex_bar();
      const T mult = sMult;
      PROF(2)
      if (a.k1) {
        const T u_w = sgd_l1 ? T(scur[1]) : T(0);
        auto update = [&](uint32_t c, T x, T th, T (&st)[NS]) {
          const bool f6 = SOLVER == FMWR_TDAP && a.tdap_zw_index;
          if (f6) (void)coord_step<T, SOLVER, true, FAST, FAST>(th, mult * x, st, sp, sp.l1, u_w);     // w refreshed below (F6)
          else th = coord_step<T, SOLVER, true, FAST, FAST>(th, mult * x, st, sp, sp.l1, u_w);
          if (has_state) {
#pragma unroll
            for (int s = 0; s < NS; ++s) a.sw[s][c] = st[s];
          }
          if (!f6) a.w[c] = th;
        };
        if (lsingle) {
#pragma unroll
          for (int q = 0; q < NL; ++q)
            if ((uint32_t)(q * 32 + lane) < nnz) update(kc[q], kx[q], kw[q], ksw[q]);
        } else {
          for (uint32_t i = lane; i < nnz; i += 32) {
            uint32_t c; T x, st[NS] = {};
            entry(i, c, x);
            const T th = a.w[c];
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) st[s] = a.sw[s][c];
            }
            update(c, x, th, st);
          }
        }
      }
      // F6: TDAP linear refresh reads z_w[position in row], not z_w[column] (TDAP_Learner.h:207).  nu_w / h_w / w are
      // written by this warp only, so a warp-level sync orders the refresh after the state updates above.
      if (SOLVER == FMWR_TDAP && a.tdap_zw_index && a.k1) {
        __syncwarp();
        if (lsingle) {                                  // column and the fresh delta_w[column] are still in registers
#pragma unroll
          for (int q = 0; q < NL; ++q) {
            const uint32_t i = q * 32 + lane;           // i < nnz(row) <= p
            if (i < nnz) {
              const T z = a.sw[1][i] - a.sw[3][i];        // z_w[pos] = nu_w[pos] - h_w[pos]
              a.w[kc[q]] = tdap_refresh<T, FAST>(z, ksw[q][2], sp.l1_w, sp.l2_w);
            }
          }
        } else {
          for (uint32_t i = lane; i < nnz; i += 32) {
            const uint32_t c = a.col[b + i];
            const T z = a.sw[1][i] - a.sw[3][i];
            a.w[c] = tdap_refresh<T, FAST>(z, a.sw[2][c], sp.l1_w, sp.l2_w);
          }
        }
      }
      PROF(3)
      ex_bar();
    } else {
      // =========================== pipeline warp ===========================
      // SGD cumulative-L1 totals advance once per sample, before the updates (SGD_Learner.h:92-97)
      if (lane == 0 && sgd_l1) { scur[1] += (double)sp.lr * (double)sp.reg_w; scur[2] += (double)sp.lr * (double)sp.reg_v; }
      uint32_t pa_row = 0, pb_b = 0, pb_e = 0, pc_col[NC];
      float pb_y = 0.f, pc_val[NC];
      if (lane == 0 && t + 4 < a.t_end) { pa_row = row_at(pos); if (++pos == period) pos = 0; }
      if (lane == 1 && t + 3 < a.t_end) {
        const uint32_t r = rRow[(t + 3) & (RING - 1)];
        pb_b = a.rowptr[r]; pb_e = a.rowptr[r + 1]; pb_y = a.y[r];
      }
      if (t + 2 < a.t_end) {
        const uint32_t b2 = rB[(t + 2) & (RING - 1)], e2 = rE[(t + 2) & (RING - 1)];
#pragma unroll
        for (int q = 0; q < NC; ++q) {
          const uint32_t idx = q * 32 + lane, j = b2 + idx;
          pc_col[q] = 0; pc_val[q] = 0.f;
          if (idx < (uint32_t)RN && j < e2) { pc_col[q] = a.col[j]; pc_val[q] = a.val[j]; }
        }
      }
      if (t + 1 < a.t_end) {
        const uint32_t n1 = min(rE[(t + 1) & (RING - 1)] - rB[(t + 1) & (RING - 1)], (uint32_t)RN);
        for (uint32_t i = lane; i < n1; i += 32) {
          const uint32_t c = rCol[(t + 1) & (CRING - 1)][i];
          const size_t off = (size_t)c * kp;
          for (int q = 0; q < kp; q += LINE) {
            prefetch_l2(a.v + off + q);
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) prefetch_l2(a.sv[s] + off + q);
            }
          }
          if (a.k1) {
            prefetch_l2(a.w + c);
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) prefetch_l2(a.sw[s] + c);
            }
          }
        }
      }
      PROF(1)
      ex_bar();
      const T mult = reduce_mult();
      PROF(2)
      ex_bar();
      if (lane == 0) {
        // scalars: w0 and its optimizer state, written to the other parity
        double s[6];
        for (int i = 0; i < 6; ++i) s[i] = scur[i];
        intercept_step<T, SOLVER, sizeof(T) == 4>(s, (double)mult, a.k0, sq_acc, sp, inv_alpha_w);
        for (int i = 0; i < 6; ++i) snext[i] = s[i];
        snext[6] = scur[6]; snext[7] = scur[7];
      }
      // run-ahead results into the rings
      if (lane == 0 && t + 4 < a.t_end) rRow[(t + 4) & (RING - 1)] = pa_row;
      if (lane == 1 && t + 3 < a.t_end) { rB[(t + 3) & (RING - 1)] = pb_b; rE[(t + 3) & (RING - 1)] = pb_e; rY[(t + 3) & (RING - 1)] = pb_y; }
      if (t + 2 < a.t_end) {
#pragma unroll
        for (int q = 0; q < NC; ++q) {
          const uint32_t idx = q * 32 + lane;
          if (idx < (uint32_t)RN) { rCol[(t + 2) & (CRING - 1)][idx] = pc_col[q]; rVal[(t + 2) & (CRING - 1)][idx] = pc_val[q]; }
        }
      }
      PROF(3)
      ex_bar();
    }
  }
#ifdef FMWR_EXACT_PROF
  if (lane == 0 && (warp == 0 || warp >= EX_FW)) {
    const long long N = a.t_end - a.t_begin;
    printf("exact prof %s: gather %lld reduce %lld [bar] mult %lld update %lld [bar]\n",
           warp == 0 ? "factor warp 0" : (warp == W_LIN ? "linear warp  " : "pipeline warp"), pt[0] / N, pt[1] / N, pt[2] / N, pt[3] / N);
  }
#endif
  if (tid < 8) a.scal[tid] = sc[a.t_end & 1][tid];
}

}  // namespace fmwr
#include "train_exact_pipe.cuh"
namespace fmwr {

template <class T, int SOLVER>
struct ExactPipeLaunch {
  fmwr_ctx* ctx; ExactArgs<T> args; double avg_nnz; bool launched; bool force;
  template <class TT, int LPR, int CH>
  void run()
  {
    const bool has_state = (SOLVER != FMWR_SGD) || args.sp.l1;
    const XpPlan pl = xp_plan<TT>(LPR * CH, 32 / LPR, has_state, solver_nst(SOLVER), avg_nnz);
    launched = false;
    if (pl.ecap < 32 / LPR) return;          // a factor row too wide to stage even one round: the CTA-wide kernel takes it
    // fp64 FTRL / TDAP are bound by the IEEE sqrt / divide sequences of the 1248 coordinate steps of a sample, not by latency: one
    // warp per sample loses to the CTA-wide kernel's 14 warps per sample there (7.8 vs 4.5 us per sample measured)
    // TDAP (five staged arrays: only 4 samples in flight, and the longest coordinate step) is a tie in fp32 (1.84 vs 1.91 us per sample)
    // and stays on the kernel whose speed does not depend on the data's column collisions
    if (((sizeof(TT) == 8 && SOLVER != FMWR_SGD) || SOLVER == FMWR_TDAP) && !force) return;
    FMWR_CUDA(cudaFuncSetAttribute(exact_pipe_kernel<TT, LPR, CH, SOLVER>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    FMWR_LAUNCH(ctx, (exact_pipe_kernel<TT, LPR, CH, SOLVER>), 1, (pl.teams + 3) * 32, pl.total, args, pl.teams, pl.ecap, pl.na,
                (uint32_t)pl.off_stage, (uint32_t)pl.stage_bytes_per_team);
    launched = true;
  }
};

template <class T, int SOLVER>
struct ExactLaunch {
  fmwr_ctx* ctx; ExactArgs<T> args;
  template <class TT, int LPR, int CH>
  void run() { FMWR_LAUNCH(ctx, (exact_kernel<TT, LPR, CH, SOLVER>), 1, EX_THREADS, 0, args); }
};

// The sample visit sequence when it is not the plain scan: the caller's explicit list, or strides of 1 + floor(U * random_step)
// drawn from glibc rand() like random_select (reference src/util/Random.h:126-132; scan loops SGD_Learner.h:84-88).  Empty result:
// the plain scan i = 1 .. n-1 (F5).  Shared by the exact and the throughput mode.
std::vector<uint32_t> visit_order_host(const fmwr_data* d, const fmwr_solver_cfg* s)
{
  std::vector<uint32_t> order_host;
  const int64_t max_iter = s->max_iter;
  if (s->visit_order && s->n_visit > 0) {
    order_host.assign(s->visit_order, s->visit_order + s->n_visit);
  } else if (s->random_step > 1) {
    auto draw = [&]() -> uint32_t { return (uint32_t)((std::rand() / ((double)RAND_MAX + 1)) * s->random_step + 1); };
    while ((int64_t)order_host.size() < max_iter) {
      const size_t before = order_host.size();
      for (uint32_t i = draw(); i < (uint32_t)d->n && (int64_t)order_host.size() < max_iter; i += draw()) order_host.push_back(i);
      if (order_host.size() == before && d->n <= 1) break;
    }
  }
  for (uint32_t r : order_host) FMWR_REQUIRE((int64_t)r < d->n, FMWR_ERR_ARG, "visit_order entry out of range");
  return order_host;
}

template <class T>
static void train_exact_t(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr,
                          const Holdout* holdout)
{
  const SolverParams<double> spd = make_params<double>(m, s);
  model_alloc_state(m, solver_state_count(spd), s->solver, s->warm_state != 0);   // Learner::init(): the state restarts at zero unless warm

  ExactArgs<T> a;
  memset(&a, 0, sizeof a);
  a.rowptr = d->rowptr.p; a.col = d->col.p; a.val = d->val.p; a.y = d->y.p;
  a.w = (T*)m->w.p; a.v = (T*)m->v.p; a.scal = (double*)m->scal.p;
  for (int i = 0; i < 4; ++i) { a.sw[i] = (T*)m->sw[i].p; a.sv[i] = (T*)m->sv[i].p; }
  a.kp = m->kp; a.k0 = m->cfg.keep_w0; a.k1 = m->cfg.keep_w1; a.task = m->cfg.task;
  a.n = d->n;
  a.skip_row0 = (s->compat & FMWR_COMPAT_SKIP_ROW0) ? 1 : 0;
  a.tdap_zw_index = (s->compat & FMWR_COMPAT_TDAP_ZW_INDEX) ? 1 : 0;
  a.sp = make_params<T>(m, s);
  a.lo = s->min_target; a.hi = s->max_target;
  { const char* nh = std::getenv("FMWR_EXACT_NOHAZARD"); a.nohazard = (nh && nh[0] == '1') ? 1 : 0; }
  bool pipelined = true;
  bool force_pipe = false;
  { const char* pp = std::getenv("FMWR_EXACT_PIPE"); if (pp && pp[0] == '0') pipelined = false; if (pp && pp[0] == '2') force_pipe = true; }
  const double avg_nnz = d->n > 0 ? (double)d->nnz / (double)d->n : 0.0;

  // visit order.  random_step == 1: the reference scans i = 1 .. n-1 (F5).  random_step > 1: strides of
  // 1 + floor(U * random_step) from glibc rand() (reference src/util/Random.h:126-132); the caller may pass
  // the sequence explicitly (visit_order) so both sides of a comparison use the same one.
  DBuf<uint32_t> order_dev;
  const int64_t max_iter = s->max_iter;
  std::vector<uint32_t> order_host = visit_order_host(d, s);
  if (!order_host.empty()) {
    order_dev.alloc(order_host.size());
    FMWR_CUDA(cudaMemcpyAsync(order_dev.p, order_host.data(), 4 * order_host.size(), cudaMemcpyHostToDevice, ctx->stream));
    a.order = order_dev.p; a.order_len = (int64_t)order_host.size();
  } else if (d->n <= a.skip_row0) return;   // no row to visit (the reference would never leave its scan loop)

  Tracker trk(ctx, m, s, tr, holdout);
  const int step = trk.step;
  int64_t iter = 0;
  while (iter < max_iter) {
    // run up to and including the next sample the tracker records: the reference evaluates after the update of samples
    // 0, step, 2*step, ... and of sample max_iter-1 (SGD_Learner.h:140-143)
    const int64_t next = step > 0 ? std::min<int64_t>((iter + step - 1) / step * step + 1, max_iter) : max_iter;
    a.t_begin = iter; a.t_end = next;
    bool launched = false;
    if (pipelined) {
      // several samples in flight, serial semantics kept by column-hazard tracking (train_exact_pipe.cuh)
      if (s->solver == FMWR_SGD) { ExactPipeLaunch<T, FMWR_SGD> L{ctx, a, avg_nnz, false, force_pipe}; dispatch_layout<T>(m->kp, L); launched = L.launched; }
      else if (s->solver == FMWR_FTRL) { ExactPipeLaunch<T, FMWR_FTRL> L{ctx, a, avg_nnz, false, force_pipe}; dispatch_layout<T>(m->kp, L); launched = L.launched; }
      else { ExactPipeLaunch<T, FMWR_TDAP> L{ctx, a, avg_nnz, false, force_pipe}; dispatch_layout<T>(m->kp, L); launched = L.launched; }
    }
    if (launched) {}
    else if (s->solver == FMWR_SGD) { ExactLaunch<T, FMWR_SGD> L{ctx, a}; dispatch_layout<T>(m->kp, L); }
    else if (s->solver == FMWR_FTRL) { ExactLaunch<T, FMWR_FTRL> L{ctx, a}; dispatch_layout<T>(m->kp, L); }
    else { ExactLaunch<T, FMWR_TDAP> L{ctx, a}; dispatch_layout<T>(m->kp, L); }
    iter = next;
    if (trk.due(iter - 1) && trk.record(iter - 1, tracker_score(ctx, m, d, s))) break;
  }
  trk.restore_best();
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  trk.write_trace(iter);
}

void train_exact(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* holdout)
{
  if (m->prec == FMWR_F64) train_exact_t<double>(ctx, m, d, s, tr, holdout);
  else train_exact_t<float>(ctx, m, d, s, tr, holdout);
}

}  // namespace fmwr
