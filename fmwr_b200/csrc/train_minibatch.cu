// Throughput (minibatch) mode of SGD / FTRL-Proximal / TDAP.
//
// The reference has no minibatch semantics (every solver is batch = 1, reference
// src/solver/*_Learner.h); this mode is DEFINED here and reduces to the exact mode at batch = 1:
//
//   for each batch of B consecutive rows (in the reference's scan order):
//     K1  row-parallel forward with frozen parameters: mult_r and S_r[f] for every row of the batch
//     K2  coordinate-parallel update: every touched coordinate c receives ONE optimizer step with the
//         summed gradient  G_c = sum_{r in batch, x_rc != 0} g_rc   (g_rc exactly as in the exact mode),
//         FTRL: n += G^2, z += G - sigma*theta; TDAP likewise; SGD: theta -= lr*G then the L2 / L1 step.
//         w0: FTRL/TDAP use the summed gradient; SGD uses the batch MEAN (a summed dense gradient
//         diverges for B*lr*0.25 > 2); identical at B = 1.
//
// K2 does not use atomics: the batch's non-zeros are pre-sorted by (batch, feature, row)
// (data.cu: minibatch_build), so one lane group owns one (batch, feature) segment, reduces its rows'
// gradients in registers and writes the coordinate once -- deterministic and contention-free.
#include "forward_stream.cuh"
#include "coord.cuh"

#include <cmath>


namespace fmwr {

void comm_allreduce_sum(fmwr_ctx* ctx, void* buf, size_t count, bool f64);

// ---- K1: forward + multiplier + S cache --------------------------------------------------------
template <class T, int LPR, int CH, int TEAM, bool PEERK>
__global__ void __launch_bounds__(256, FWD_BLOCKS)
mb_forward_kernel(const uint32_t* __restrict__ rowptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
                  const float* __restrict__ y, const T* __restrict__ w, const T* __restrict__ v,
                  const double* __restrict__ scal, int kp, int k0, int k1, int task, T lo, T hi,
                  int64_t row_begin, int rows, T* __restrict__ mult, T* __restrict__ Scache, int s_stride, int partial, PeerArgs pa)
{
  typedef typename Vec<T>::type V16;
  constexpr int TPW = 32 / TEAM;
  const int lane = threadIdx.x & 31;
  const int tl = lane % TEAM;
  const int warp0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int step = gridDim.x * (blockDim.x >> 5) * TPW;
  const T w0 = T(scal[0]);
  for (int base = warp0 * TPW; base < rows; base += step) {       // uniform per warp: every lane reaches the shuffles
    const int r = base + lane / TEAM;
    const int64_t row = row_begin + r;
    uint32_t b = 0u, e = 0u;
    if (r < rows) { b = __ldg(rowptr + row); e = __ldg(rowptr + row + 1); }
    T S[CH][Vec<T>::N];
    if (!partial) {
      const T score = team_forward<T, LPR, CH, TEAM>(col, val, b, e, w, v, kp, w0, k0, k1, S);
      if (tl == 0 && r < rows) mult[r] = grad_mult_fast(task, score, T(__ldg(y + row)), lo, hi);
    } else {
      // feature-parallel: this rank holds a column slice, so the row's score is not known yet.  Emit the partials:
      // S_f of the slice and its additive scalar (see team_gather); 1/2 sum S_f^2 is formed after the exchange
      const T addend = team_forward_partial<T, LPR, CH, TEAM>(col, val, b, e, w, v, kp, k1, S);
      if (PEERK) {
        // peer window: the partial goes straight into the memory of the rank that finalises this row (NVLink stores)
        if (r < rows) {
          const int owner = r / pa.rows_per_owner;
          T* dst = reinterpret_cast<T*>(peer_base(pa, owner) + pa.off_P) + ((size_t)pa.rank * pa.rows_per_owner + (r - owner * pa.rows_per_owner)) * s_stride;
          if (tl == 0) {                      // a whole 16-byte vector {addend, 0..}: no partial-sector write over NVLink
            T pad[Vec<T>::N];
#pragma unroll
            for (int i = 0; i < Vec<T>::N; ++i) pad[i] = T(0);
            pad[0] = addend;
            *reinterpret_cast<V16*>(dst + kp) = arr_to_vec(pad);
          }
          if (tl < LPR) {
#pragma unroll
            for (int ch = 0; ch < CH; ++ch) reinterpret_cast<V16*>(dst)[ch * LPR + tl] = arr_to_vec(S[ch]);
          }
        }
        continue;
      }
      if (tl == 0 && r < rows) Scache[(size_t)r * s_stride + kp] = addend;
    }
    if (tl < LPR && r < rows) {
      V16* dst = reinterpret_cast<V16*>(Scache + (size_t)r * s_stride);
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) dst[ch * LPR + tl] = arr_to_vec(S[ch]);
    }
  }
  if (PEERK) peer_signal(pa, PEER_FLAG1, PEER_EPOCH1, PEER_COUNT1);
}

// ---- peer exchange: the rank that owns a row sums the world's partials IN RANK ORDER (deterministic), forms the
// score and the multiplier, and stores the row [S_f totals (kp), multiplier, 0...] into every rank's S cache.
// One LPR-lane group per row (32/LPR rows per warp), 16-byte loads and stores throughout. -------------------------
template <class T, int LPR, int CH>
__global__ void __launch_bounds__(256)
mb_exchange_kernel(const float* __restrict__ y, const double* __restrict__ scal, int kp, int k0, int task, T lo, T hi,
                   int64_t row_begin, int rows, int s_stride, PeerArgs pa)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int G = 32 / LPR;
  peer_wait(pa, PEER_FLAG1, PEER_EPOCH1);
  const int lane = threadIdx.x & 31;
  const int g = lane / LPR, l = lane % LPR;
  const int grp0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * G + g;
  const int ngrp = gridDim.x * (blockDim.x >> 5) * G;
  const int r_lo = pa.rank * pa.rows_per_owner;
  const int r_hi = min(rows, r_lo + pa.rows_per_owner);
  const int n_local = max(0, r_hi - r_lo);
  const T* P = reinterpret_cast<const T*>(peer_base(pa, pa.rank) + pa.off_P);
  const T w0 = k0 ? T(scal[0]) : T(0);
  for (int base = 0; base < n_local; base += ngrp) {             // warp-uniform trip count: the shuffles below need every lane
    const int rl = base + grp0;
    const bool ok = rl < n_local;
    const int r = r_lo + rl;
    T S[CH][VN];
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int i = 0; i < VN; ++i) S[ch][i] = T(0);
    T add = T(0);
    if (ok) {
      for (int h = 0; h < pa.world; ++h) {
        const T* row = P + ((size_t)h * pa.rows_per_owner + rl) * s_stride;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) {
          T t[VN];
          vec_to_arr(reinterpret_cast<const V16*>(row)[ch * LPR + l], t);
#pragma unroll
          for (int i = 0; i < VN; ++i) S[ch][i] += t[i];
        }
        if (l == 0) add += row[kp];
      }
    }
    T acc = add;
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int i = 0; i < VN; ++i) acc += T(0.5) * S[ch][i] * S[ch][i];
    acc = team_sum<T, LPR>(acc);
    if (ok) {
      const T m = grad_mult_fast(task, w0 + acc, T(__ldg(y + row_begin + r)), lo, hi);
      T tail[VN];
#pragma unroll
      for (int i = 0; i < VN; ++i) tail[i] = T(0);
      tail[0] = m;
#pragma unroll
      for (int h = 0; h < 8; ++h) {
        if (h >= pa.world) break;
        T* dst = reinterpret_cast<T*>(pa.base[h] + pa.off_S) + (size_t)r * s_stride;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) reinterpret_cast<V16*>(dst)[ch * LPR + l] = arr_to_vec(S[ch]);
        if (l == 0) {
          *reinterpret_cast<V16*>(dst + kp) = arr_to_vec(tail);
          reinterpret_cast<T*>(pa.base[h] + pa.off_mult)[r] = m;     // compact copy: the intercept block of K2 sums these with unit stride
        }
      }
    }
  }
  peer_signal(pa, PEER_FLAG2, PEER_EPOCH2, PEER_COUNT2);
}

// after the all-reduce: score = w0 + addend + 1/2 sum_f S_f^2 ; one warp per row
template <class T>
__global__ void __launch_bounds__(256)
mb_finalize_kernel(const float* __restrict__ y, const double* __restrict__ scal, int kp, int k0, int task, T lo, T hi,
                   int64_t row_begin, int rows, const T* __restrict__ Scache, int s_stride, T* __restrict__ mult)
{
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const T* row = Scache + (size_t)r * s_stride;
  T acc = T(0);
  for (int f = lane; f < kp; f += 32) { const T s = row[f]; acc += T(0.5) * s * s; }
  acc = warp_sum(acc);
  if (lane == 0) {
    const T score = (k0 ? T(scal[0]) : T(0)) + row[kp] + acc;
    mult[r] = grad_mult<T>(task, score, T(__ldg(y + row_begin + r)), lo, hi);
  }
}

// tracker on a feature-sharded model: summed partials -> score -> link -> prediction (one warp per row)
template <class T>
__global__ void __launch_bounds__(256)
mb_score_kernel(const double* __restrict__ scal, int kp, int k0, int rows, const T* __restrict__ Scache, int s_stride, int link, double lo, double hi,
                const double* __restrict__ pnY, double* __restrict__ out)
{
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const T* row = Scache + (size_t)r * s_stride;
  T acc = T(0);
  for (int f = lane; f < kp; f += 32) { const T sv = row[f]; acc += T(0.5) * sv * sv; }
  acc = warp_sum(acc);
  if (lane == 0) out[r] = apply_link(link, (double)((k0 ? T(scal[0]) : T(0)) + row[kp] + acc), lo, hi, pnY);
}

// ---- K2: one lane group per (batch, feature) segment --------------------------------------------
template <class T>
struct MbUpdArgs {
  const uint32_t* seg_ptr; const uint4* seg_rec; const uint32_t* ent_row; const float* ent_val;
  uint32_t seg_begin, seg_end;
  int64_t row_begin; int rows;          // rows of this batch that take part (row filter for a truncated last batch)
  const T* mult; const T* Scache;
  T* w; T* v; double* scal;
  T* sw[4]; T* sv[4];
  int kp, k0, k1, s_stride;
  SolverParams<T> sp;
  T u_w, u_v;                           // SGD cumulative-L1 totals after this batch
  int mult_stride;                      // 1, or the S-cache row stride when the multiplier lives in the row's padding (peer mode)
  int peer;                             // peer-window exchange: wait for every rank's row totals first
  const double* msum; int msum_n;       // fused exchange: the ranks' sums of multipliers (else the intercept block sums a.mult itself)
  const T* mult_compact;                // unfused peer exchange: the multipliers once more with unit stride (a.mult is strided there)
  PeerArgs pa;
};

template <int SOLVER> struct K2Tune { enum { BLOCKS = SOLVER == FMWR_TDAP ? 3 : 5, UE = SOLVER == FMWR_TDAP ? 4 : 2 }; };

// the intercept (dense coordinate): fixed-order reduction of the batch's multipliers by ONE block.  It is block 0 so
// that its serial chain of loads overlaps the rest of the grid instead of forming the kernel's tail.
template <class T, int SOLVER>
__device__ __forceinline__ void mb_intercept(const MbUpdArgs<T>& a)
{
  const SolverParams<T>& sp = a.sp;
  __shared__ double red[32];
  double acc = 0.0;
  const int nt = (int)blockDim.x;
  if (a.msum) {
    if (threadIdx.x == 0) for (int i = 0; i < a.msum_n; ++i) acc += a.msum[i];      // rank order: every rank forms the same sum
  } else {
    constexpr int UN = 16;
    const T* mp = a.mult_compact ? a.mult_compact : a.mult;
    const size_t ms = a.mult_compact ? 1 : (size_t)a.mult_stride;
    int r = threadIdx.x;
    for (; r + (UN - 1) * nt < a.rows; r += UN * nt) {
      T t[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) t[u] = mp[(size_t)(r + u * nt) * ms];
#pragma unroll
      for (int u = 0; u < UN; ++u) acc += (double)t[u];
    }
    for (; r < a.rows; r += nt) acc += (double)mp[(size_t)r * ms];
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double gsum = 0;
    for (int i = 0; i < (nt >> 5); ++i) gsum += red[i];
    double s[6];
    for (int i = 0; i < 6; ++i) s[i] = a.scal[i];
    double sq = SOLVER == FMWR_SGD ? 0.0 : sqrt(SOLVER == FMWR_FTRL ? s[2] : s[1]);
    intercept_step<T, SOLVER, false>(s, SOLVER == FMWR_SGD ? gsum / (double)a.rows : gsum, a.k0, sq, sp);
    for (int i = 0; i < 6; ++i) a.scal[i] = s[i];
  }
}

// Everything a segment needs that depends only on its 16-byte record {feature, length, first row, first value}:
// the parameter row, its optimizer state, the first row's S-cache line and multiplier, and the next LPR entries
// of the segment (lane l fetches entry 1 + l).  seg_issue requests all of it in one go; seg_finish consumes it.
template <class T, int CH, int SOLVER>
struct SegStage {
  typename Vec<T>::type th[CH], s0[CH], st[solver_nst(SOLVER)][CH];
  T m0, tw, stw[solver_nst(SOLVER)];
  uint32_t c, len, eb, r0, my_r;
  float x0, my_x;
  bool live;
};

template <class T, int LPR, int CH, int SOLVER, bool L1>
__device__ __forceinline__ void seg_issue(const MbUpdArgs<T>& a, const uint4 rec, const uint32_t eb, const int l, bool live,
                                          SegStage<T, CH, SOLVER>& sg)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NST = solver_nst(SOLVER);
  constexpr bool USE_STATE = SOLVER != FMWR_SGD || L1;
  sg.c = rec.x; sg.len = rec.y; sg.eb = eb; sg.x0 = __uint_as_float(rec.w);
  sg.r0 = rec.z - (uint32_t)a.row_begin;
  live = live && sg.r0 < (uint32_t)a.rows;        // rows ascend inside a segment: r0 outside = nothing of it in the (truncated) batch
  sg.live = live;
  sg.my_r = 0xffffffffu;                          // sentinel: (0xffffffff - row_begin) is never < rows
  sg.my_x = 0.f;
  sg.tw = T(0); sg.m0 = T(0);
#pragma unroll
  for (int st = 0; st < NST; ++st) sg.stw[st] = T(0);
  if (!live) return;
  const size_t off = (size_t)sg.c * a.kp + l * VN;
  const T* sbase = a.Scache + l * VN + sg.r0 * (uint32_t)a.s_stride;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    sg.th[ch] = reinterpret_cast<const V16*>(a.v + off)[ch * LPR];
    sg.s0[ch] = reinterpret_cast<const V16*>(sbase)[ch * LPR];
    if (USE_STATE) {
#pragma unroll
      for (int st = 0; st < NST; ++st) sg.st[st][ch] = reinterpret_cast<const V16*>(a.sv[st] + off)[ch * LPR];
    }
  }
  sg.m0 = a.mult[sg.r0 * (uint32_t)a.mult_stride];
  if (a.k1 && l == 0) {
    sg.tw = a.w[sg.c];
    if (USE_STATE) {
#pragma unroll
      for (int st = 0; st < NST; ++st) sg.stw[st] = a.sw[st][sg.c];
    }
  }
  if (1u + (uint32_t)l < sg.len) { sg.my_r = __ldg(a.ent_row + eb + 1 + l); sg.my_x = __ldg(a.ent_val + eb + 1 + l); }
}

template <class T, int LPR, int CH, int SOLVER, bool L1>
__device__ __forceinline__ void seg_finish(const MbUpdArgs<T>& a, const int g, const int l, SegStage<T, CH, SOLVER>& sg)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NST = solver_nst(SOLVER);
  constexpr bool USE_STATE = SOLVER != FMWR_SGD || L1;
  constexpr bool FAST = sizeof(T) == 4;
  if (!sg.live) return;
  const uint32_t c = sg.c, len = sg.len, eb = sg.eb;
  const uint32_t rb32 = (uint32_t)a.row_begin, nrows = (uint32_t)a.rows;
  const size_t off = (size_t)c * a.kp + l * VN;
  const T* sbase = a.Scache + l * VN;
  const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));
  uint32_t my_r = sg.my_r;
  float my_x = sg.my_x;

  T th[CH][VN], Gv[CH][VN], Gw, bsum;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) vec_to_arr(sg.th[ch], th[ch]);
  seg_grad_entry<SOLVER, true>(Gw, bsum, Gv, th, sg.m0, T(sg.x0), sg.s0);
  for (uint32_t base = 1; base < len; base += LPR) {
    if (base > 1) {
      my_r = 0xffffffffu; my_x = 0.f;
      if (base + (uint32_t)l < len) { my_r = __ldg(a.ent_row + eb + base + l); my_x = __ldg(a.ent_val + eb + base + l); }
    }
    const int cnt = (int)min((uint32_t)LPR, len - base);
    constexpr int UE = LPR < K2Tune<SOLVER>::UE ? LPR : K2Tune<SOLVER>::UE;
    for (int j0 = 0; j0 < cnt; j0 += UE) {
      T xe[UE], me[UE];
      V16 se[UE][CH];
#pragma unroll
      for (int u = 0; u < UE; ++u) {
        const int src = g * LPR + j0 + u;
        const uint32_t rl = __shfl_sync(gmask, my_r, src) - rb32;
        xe[u] = T(__shfl_sync(gmask, my_x, src));
        const bool ok = rl < nrows;                // false for the padding lanes and for rows past a truncated batch
        me[u] = ok ? a.mult[rl * (uint32_t)a.mult_stride] : T(0);
        const T* sr = sbase + (ok ? rl : 0u) * (uint32_t)a.s_stride;
#pragma unroll
        for (int ch = 0; ch < CH; ++ch) se[u][ch] = reinterpret_cast<const V16*>(sr)[ch * LPR];
      }
#pragma unroll
      for (int u = 0; u < UE; ++u) seg_grad_entry<SOLVER>(Gw, bsum, Gv, th, me[u], xe[u], se[u]);
    }
  }
  seg_grad_close<SOLVER>(Gv, th, bsum);

  // ---- linear weight (lane 0 of the group)
  if (a.k1 && l == 0) {
    a.w[c] = coord_step<T, SOLVER, true, FAST, false>(sg.tw, Gw, sg.stw, a.sp, L1, a.u_w);
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) a.sw[k][c] = sg.stw[k];
    }
  }
  // ---- factors
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    T st[NST][VN] = {};
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) vec_to_arr(sg.st[k][ch], st[k]);
    }
    coord_step<T, SOLVER, false, FAST, false>(th[ch], Gv[ch], st, a.sp, L1, a.u_v);
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) reinterpret_cast<V16*>(a.sv[k] + off)[ch * LPR] = arr_to_vec(st[k]);
    }
    reinterpret_cast<V16*>(a.v + off)[ch * LPR] = arr_to_vec(th[ch]);
  }
}

// One lane group per segment.  Measured on B200 (profiles/r01_summary.md): occupancy beats per-warp depth here -- a
// 48-register build (5 resident CTAs/SM walking the segments grid-stride, entries taken two at a time) beats both the
// 40-register/6-CTA build (spills) and a software-pipelined variant with three segments in flight per group.
// TDAP carries 4 state rows and keeps 80 registers.

template <class T, int LPR, int CH, int SOLVER, bool L1>
__global__ void __launch_bounds__(256, (sizeof(T) == 4 && CH == 1) ? K2Tune<SOLVER>::BLOCKS : 1) mb_update_kernel(MbUpdArgs<T> a)
{
  constexpr int G = 32 / LPR;
  if (a.peer) peer_wait(a.pa, PEER_FLAG2, PEER_EPOCH2);
  if (blockIdx.x == 0) { mb_intercept<T, SOLVER>(a); return; }
  const int lane = threadIdx.x & 31;
  const int g = lane / LPR, l = lane % LPR;
  // grid-stride over the batch's segments: with a grid of (resident CTAs) the warps stay on the SM for the whole launch
  // instead of being re-created every 4 segments
  const uint32_t stride = (gridDim.x - 1) * (blockDim.x >> 5) * G;
  for (uint32_t seg = a.seg_begin + ((blockIdx.x - 1) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * G + g; seg < a.seg_end; seg += stride) {
    const uint4 rec = __ldg(a.seg_rec + seg);
    const uint32_t eb = __ldg(a.seg_ptr + seg);
    SegStage<T, CH, SOLVER> sg;
    seg_issue<T, LPR, CH, SOLVER, L1>(a, rec, eb, l, true, sg);
    seg_finish<T, LPR, CH, SOLVER, L1>(a, g, l, sg);
  }
}

}  // namespace fmwr
#include "update_tma.cuh"
namespace fmwr {

// ---- K2, dense variant (update_tma.cuh): producer warp + 8 consumer warps over a ring of TMA-filled stages ----------------
template <class T, int LPR, int CH, int SOLVER, bool L1, int TS, int NS, int MINB>
__global__ void __launch_bounds__(TM_THREADS, MINB) mb_update_tma_kernel(MbUpdArgs<T> a)
{
  typedef TmGeom<T, LPR, CH, SOLVER, L1, TS, NS> G;
  constexpr int GRP = 32 / LPR;                         // lane groups (segments) per warp
  constexpr int NSTW = solver_nst(SOLVER);
  extern __shared__ __align__(128) unsigned char tm_smem[];
  unsigned char* stages = tm_smem;
  uint32_t* hdr_all = reinterpret_cast<uint32_t*>(tm_smem + NS * G::STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tm_smem + NS * G::STAGE_BYTES + NS * G::HDR_WORDS * 4);   // full[NS], done[NS]
  if (a.peer) peer_wait(a.pa, PEER_FLAG2, PEER_EPOCH2);
  if (blockIdx.x == 0) { mb_intercept<T, SOLVER>(a); return; }
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(smem_u32(bars + s), 1u); mbar_init(smem_u32(bars + NS + s), TM_CONS_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t n_seg = a.seg_end - a.seg_begin;
  const uint32_t n_tiles = (n_seg + TS - 1) / TS;
  const uint32_t first = blockIdx.x - 1, stride = gridDim.x - 1;
  const uint32_t my_tiles = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0u;

  if (warp == TM_CONS_WARPS) {
    // ================================ producer: loads and write-backs, lane 0 only =================================
    if (lane != 0) return;
    const uint64_t pol = l2_policy();
    uint32_t wb_c0[NS], wb_rows[NS];                      // pending write-back of each stage (rows == 0: none)
#pragma unroll
    for (int s = 0; s < NS; ++s) { wb_c0[s] = 0u; wb_rows[s] = 0u; }
    auto write_back = [&](int s) {
      unsigned char* st = stages + (size_t)s * G::STAGE_BYTES;
      const uint32_t c0 = wb_c0[s], nr = wb_rows[s];
      if (nr) {
        const uint32_t bytes = nr * G::ROWB;
        bulk_s2g(reinterpret_cast<unsigned char*>(a.v) + (size_t)c0 * G::ROWB, smem_u32(st + G::OFF_PAR), bytes, pol);
        if (G::USE_STATE) {
#pragma unroll
          for (int i = 0; i < NSTW; ++i)
            bulk_s2g(reinterpret_cast<unsigned char*>(a.sv[i]) + (size_t)c0 * G::ROWB, smem_u32(st + G::OFF_PAR + (i + 1) * G::RMAX * G::ROWB), bytes, pol);
        }
        bulk_commit();
        bulk_wait_read0();                                 // the stage may be refilled once the stores have READ it
      }
    };
    // the tile's extent (first / last feature, first / one-past-last entry) comes from four scattered words: fetched one
    // tile ahead so their latency never sits between a freed stage and its refill
    uint32_t d_c0 = 0u, d_c1 = 0u, d_e0 = 0u, d_e1 = 0u;
    auto fetch_desc = [&](uint32_t i) {
      if (i >= my_tiles) return;
      const uint32_t s0 = a.seg_begin + (first + i * stride) * TS;
      const uint32_t ns = min((uint32_t)TS, a.seg_end - s0);
      d_c0 = __ldg(&a.seg_rec[s0].x); d_c1 = __ldg(&a.seg_rec[s0 + ns - 1].x);
      d_e0 = __ldg(a.seg_ptr + s0); d_e1 = __ldg(a.seg_ptr + s0 + ns);
    };
    fetch_desc(0);
    for (uint32_t i = 0; i < my_tiles; ++i) {
      const int s = (int)(i % NS);
      unsigned char* st = stages + (size_t)s * G::STAGE_BYTES;
      uint32_t* hdr = hdr_all + s * G::HDR_WORDS;
      const uint32_t c0 = d_c0, c1 = d_c1, e0 = d_e0, e1 = d_e1;
      fetch_desc(i + 1);
      if (i >= NS) {
        mbar_wait(smem_u32(bars + NS + s), ((i / NS) - 1) & 1u);     // consumers are done with the tile that lived here
        write_back(s);
      }
      const uint32_t t = first + i * stride;
      const uint32_t s0 = a.seg_begin + t * TS;
      const uint32_t ns = min((uint32_t)TS, a.seg_end - s0);
      const uint32_t nrows = c1 - c0 + 1u;
      const uint32_t s0a = s0 & ~3u, e0a = e0 & ~3u, c0a = c0 & ~3u;
      const uint32_t nsp = ((s0 + ns + 1u) - s0a + 3u) & ~3u;          // seg_ptr words [s0a, s0 + ns], rounded to 16 bytes
      const uint32_t nen = (e1 - e0a + 3u) & ~3u;
      const uint32_t nw = ((c1 + 1u) - c0a + 3u) & ~3u;
      const bool dense = nrows <= (uint32_t)G::RMAX && nen <= (uint32_t)G::EMAX + 8u;
      hdr[0] = dense ? 1u : 0u; hdr[1] = c0; hdr[2] = nrows; hdr[3] = s0 - s0a; hdr[4] = e0; hdr[5] = e0 - e0a; hdr[6] = c0 - c0a; hdr[7] = ns;
      const uint32_t full = smem_u32(bars + s);
      uint32_t tx = ns * 16u + nsp * 4u;
      bulk_g2s(smem_u32(st + G::OFF_REC), a.seg_rec + s0, ns * 16u, full, pol);
      bulk_g2s(smem_u32(st + G::OFF_SEGP), a.seg_ptr + s0a, nsp * 4u, full, pol);
      wb_rows[s] = 0u;
      if (dense) {
        if (nen) {
          bulk_g2s(smem_u32(st + G::OFF_EROW), a.ent_row + e0a, nen * 4u, full, pol);
          bulk_g2s(smem_u32(st + G::OFF_EVAL), a.ent_val + e0a, nen * 4u, full, pol);
          tx += 2u * nen * 4u;
        }
        const uint32_t pbytes = nrows * G::ROWB;
        bulk_g2s(smem_u32(st + G::OFF_PAR), reinterpret_cast<const unsigned char*>(a.v) + (size_t)c0 * G::ROWB, pbytes, full, pol);
        tx += pbytes;
        if (G::USE_STATE) {
#pragma unroll
          for (int k = 0; k < NSTW; ++k) {
            bulk_g2s(smem_u32(st + G::OFF_PAR + (k + 1) * G::RMAX * G::ROWB), reinterpret_cast<const unsigned char*>(a.sv[k]) + (size_t)c0 * G::ROWB, pbytes, full, pol);
            tx += pbytes;
          }
        }
        if (a.k1) {
          const uint32_t wbytes = nw * (uint32_t)sizeof(T);
          bulk_g2s(smem_u32(st + G::OFF_W), a.w + c0a, wbytes, full, pol);
          tx += wbytes;
          if (G::USE_STATE) {
#pragma unroll
            for (int k = 0; k < NSTW; ++k) {
              bulk_g2s(smem_u32(st + G::OFF_W + (k + 1) * (G::RMAX + 8) * (int)sizeof(T)), a.sw[k] + c0a, wbytes, full, pol);
              tx += wbytes;
            }
          }
        }
        wb_c0[s] = c0; wb_rows[s] = nrows;
      }
      mbar_arrive_expect_tx(full, tx);
    }
    // drain: write back what the consumers are still working on
    for (uint32_t i = (my_tiles > (uint32_t)NS ? my_tiles - NS : 0u); i < my_tiles; ++i) {
      const int s = (int)(i % NS);
      mbar_wait(smem_u32(bars + NS + s), (i / NS) & 1u);
      write_back(s);
    }
    bulk_wait0();
    return;
  }

  // ==================================== consumers ====================================================================
  const int g = lane / LPR, l = lane % LPR;
  for (uint32_t i = 0; i < my_tiles; ++i) {
    const int s = (int)(i % NS);
    unsigned char* st = stages + (size_t)s * G::STAGE_BYTES;
    const uint32_t* hdr = hdr_all + s * G::HDR_WORDS;
    mbar_wait(smem_u32(bars + s), (i / NS) & 1u);
    const int ns = (int)hdr[7];
    if (hdr[0]) {
      for (int j = warp * GRP + g; j < ns; j += TM_CONS_WARPS * GRP) seg_dense<T, LPR, CH, SOLVER, L1, G>(a, st, hdr, j, l);
      fence_proxy_async();                               // this thread's shared-memory writes -> visible to the bulk stores
    } else {
      // sparse tile: the gather path of mb_update_kernel, records and offsets from the stage
      for (int j0 = warp * GRP; j0 < ns; j0 += TM_CONS_WARPS * GRP) {      // warp-uniform trip count (seg_finish shuffles)
        const int j = j0 + g;
        const bool live = j < ns;
        const uint4 rec = live ? reinterpret_cast<const uint4*>(st + G::OFF_REC)[j] : make_uint4(0u, 0u, 0xffffffffu, 0u);
        const uint32_t eb = live ? reinterpret_cast<const uint32_t*>(st + G::OFF_SEGP)[hdr[3] + j] : 0u;
        SegStage<T, CH, SOLVER> sg;
        seg_issue<T, LPR, CH, SOLVER, L1>(a, rec, eb, l, live, sg);
        seg_finish<T, LPR, CH, SOLVER, L1>(a, g, l, sg);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(bars + NS + s));
  }
}

template <class T>
struct MbLaunch {
  fmwr_ctx* ctx; fmwr_model* m; fmwr_data* d; const fmwr_solver_cfg* s;
  int64_t row_begin; int rows; T* mult; T* Scache; MbUpdArgs<T> ua; int phase;   // phase 0: K1, 1: K2
  int s_stride; int partial; PeerArgs pa; bool fused_exchange = false;
  template <class TT, int LPR, int CH, int TEAM> void k1();
  void k1_stream()
  {
    SfArgs a;
    memset(&a, 0, sizeof a);
    a.rowptr = d->rowptr.p; a.col = d->col.p; a.val = d->val.p; a.y = d->y.p; a.w = (const float*)m->w.p; a.v = (const float*)m->v.p;
    a.scal = (const double*)m->scal.p; a.k0 = m->cfg.keep_w0; a.k1 = m->cfg.keep_w1; a.task = m->cfg.task;
    a.lo = (float)s->min_target; a.hi = (float)s->max_target; a.row_begin = row_begin; a.rows = rows;
    a.mult = (float*)mult; a.Scache = (float*)Scache; a.s_stride = s_stride; a.pa = pa;
    a.debug = getenv("FMWR_PEER_DEBUG") != nullptr;
    const int grid = stream_grid(ctx, rows, &a.rpg);
    if (partial == 2) FMWR_LAUNCH(ctx, forward_stream_kernel<SF_PARTIAL_PEER>, grid, 256, 0, a);
    else if (partial == 1) FMWR_LAUNCH(ctx, forward_stream_kernel<SF_PARTIAL>, grid, 256, 0, a);
    else FMWR_LAUNCH(ctx, forward_stream_kernel<SF_TRAIN>, grid, 256, 0, a);
  }
  template <class TT, int LPR, int CH, int SOLVER, bool L1, int TS, int NS, int MINB>
  void tma_launch(uint32_t nseg)
  {
    typedef TmGeom<TT, LPR, CH, SOLVER, L1, TS, NS> G;
    static int occ = 0;                                   // resident CTAs per SM of this instantiation
    if (!occ) {
      FMWR_CUDA(cudaFuncSetAttribute(mb_update_tma_kernel<TT, LPR, CH, SOLVER, L1, TS, NS, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM_BYTES));
      int o = 0;
      FMWR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, mb_update_tma_kernel<TT, LPR, CH, SOLVER, L1, TS, NS, MINB>, TM_THREADS, (size_t)G::SMEM_BYTES));
      occ = o < 1 ? 1 : o;
    }
    const int64_t n_tiles = ceil_div64((int64_t)nseg, TS);
    const int grid = (int)std::min<int64_t>(n_tiles, (int64_t)ctx->sm_count * occ) + 1;     // +1: the intercept block
    FMWR_LAUNCH(ctx, (mb_update_tma_kernel<TT, LPR, CH, SOLVER, L1, TS, NS, MINB>), grid, TM_THREADS, (size_t)G::SMEM_BYTES, ua);
  }
  template <class TT, int LPR, int CH>
  void tma(uint32_t nseg)
  {
    switch (s->solver) {
      case FMWR_SGD:
        if (ua.sp.l1) tma_launch<TT, LPR, CH, FMWR_SGD, true, 32, 3, 3>(nseg);
        else tma_launch<TT, LPR, CH, FMWR_SGD, false, 32, 3, 3>(nseg);
        break;
      case FMWR_FTRL:
        // measured on configs[1] (profiles/r02_summary.md): 32-segment tiles, 3 stages, 3 CTAs/SM 168 us per batch; 2 stages 180;
        // 4 CTAs/SM (56 registers, spills) 204; 64-segment tiles x 2 stages x 2 CTAs 184; the gather kernel 178
        tma_launch<TT, LPR, CH, FMWR_FTRL, false, 32, 3, 3>(nseg);
        break;
      default: tma_launch<TT, LPR, CH, FMWR_TDAP, false, 32, 2, 2>(nseg); break;
    }
  }
  template <class TT, int LPR, int CH>
  void run()
  {
    if (phase == 2) {
      constexpr int G = 32 / LPR;
      const int xgrid = (int)std::min<int64_t>(ceil_div(pa.rows_per_owner, 8 * G), (int64_t)ctx->sm_count * 4);
      FMWR_LAUNCH(ctx, (mb_exchange_kernel<TT, LPR, CH>), xgrid, 256, 0, d->y.p, (const double*)m->scal.p, m->kp, m->cfg.keep_w0,
                  m->cfg.task, TT(s->min_target), TT(s->max_target), row_begin, rows, s_stride, pa);
    } else if (phase == 0) {
      if (sizeof(TT) == 4 && (partial == 2 ? fused_exchange : stream_forward_ok(m, d->nnz, d->n, partial ? 2 : 8))) { k1_stream(); return; }
      const int tm = team_mode(d->nnz, d->n, LPR);
      if (tm == 1) k1<TT, LPR, CH, LPR>();
      else if (tm == 2) k1<TT, LPR, CH, (LPR <= 8 ? 16 : 32)>();
      else k1<TT, LPR, CH, 32>();
    } else {
      constexpr int G = 32 / LPR;
      const uint32_t nseg = ua.seg_end - ua.seg_begin;
      int grid = ceil_div((int64_t)nseg, 8 * G) + 1;       // +1: the intercept block
      // one wave of resident CTAs; feature-parallel ranks hold a fraction of the segments: there the one-shot grid measured
      // faster (N = 2/4/8)
      if (!(ctx->nccl_comm && ctx->world > 1)) {
        const int resident = (sizeof(TT) == 4 && CH == 1) ? (s->solver == FMWR_TDAP ? K2Tune<FMWR_TDAP>::BLOCKS : K2Tune<FMWR_SGD>::BLOCKS) : 2;
        grid = std::min(grid, ctx->sm_count * resident + 1);
      }
      // dense variant (update_tma.cuh): fp32, one 16-byte vector per lane, rows of at most 128 bytes; FMWR_K2_GATHER=1 keeps the
      // original gather kernel for every tile
      if constexpr (sizeof(TT) == 4 && CH == 1 && LPR <= 8) {
        const bool no_tma = getenv("FMWR_K2_GATHER") != nullptr;     // read per launch: tests flip it between calls
        if (!no_tma) { tma<TT, LPR, CH>(nseg); return; }
      }
      switch (s->solver) {
        case FMWR_SGD:
          if (ua.sp.l1) FMWR_LAUNCH(ctx, (mb_update_kernel<TT, LPR, CH, FMWR_SGD, true>), grid, 256, 0, ua);
          else FMWR_LAUNCH(ctx, (mb_update_kernel<TT, LPR, CH, FMWR_SGD, false>), grid, 256, 0, ua);
          break;
        case FMWR_FTRL: FMWR_LAUNCH(ctx, (mb_update_kernel<TT, LPR, CH, FMWR_FTRL, false>), grid, 256, 0, ua); break;
        default: FMWR_LAUNCH(ctx, (mb_update_kernel<TT, LPR, CH, FMWR_TDAP, false>), grid, 256, 0, ua); break;
      }
    }
  }
};

template <class T>
template <class TT, int LPR, int CH, int TEAM>
void MbLaunch<T>::k1()
{
  const int rpb = 8 * (32 / TEAM);
  // 4 resident CTAs per SM: measured best (persistent warps); peer mode wants few fat CTAs too, because each CTA ends with one
  // release fence that waits for its NVLink stores
  const int fgrid = (int)std::min<int64_t>(ceil_div(rows, rpb), (int64_t)ctx->sm_count * 4);
  // (the peer-window variant is a separate instantiation: indexing the window table by owner costs every thread a stack frame)
  if (partial == 2)
    FMWR_LAUNCH(ctx, (mb_forward_kernel<TT, LPR, CH, TEAM, true>), fgrid, 256, 0, d->rowptr.p, d->col.p, d->val.p, d->y.p,
                (const TT*)m->w.p, (const TT*)m->v.p, (const double*)m->scal.p, m->kp, m->cfg.keep_w0, m->cfg.keep_w1,
                m->cfg.task, TT(s->min_target), TT(s->max_target), row_begin, rows, mult, Scache, s_stride, partial, pa);
  else
    FMWR_LAUNCH(ctx, (mb_forward_kernel<TT, LPR, CH, TEAM, false>), fgrid, 256, 0, d->rowptr.p, d->col.p, d->val.p, d->y.p,
                (const TT*)m->w.p, (const TT*)m->v.p, (const double*)m->scal.p, m->kp, m->cfg.keep_w0, m->cfg.keep_w1,
                m->cfg.task, TT(s->min_target), TT(s->max_target), row_begin, rows, mult, Scache, s_stride, partial, pa);
}

// Tracker on a feature-sharded model (reference: the full predict_batch + metric inside the epoch, src/solver/SGD_Learner.h:140-166).
// Nothing is gathered: every rank forwards ITS column slice over all rows in chunks, the chunk's partials (S_f, additive scalar) are
// summed over the ranks, and every rank finishes score -> link -> metric on the identical totals, so all ranks record the same value.
template <class T>
static double tracker_score_sharded(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s)
{
  const int64_t n = d->n;
  const int s_stride = m->kp + 4;
  const int64_t chunk = 65536;
  DBuf<T> buf;
  buf.alloc((size_t)chunk * s_stride);
  buf.zero(ctx->stream);
  d->pred64.ensure(n);
  d->pred_prec = FMWR_F64;
  const int link = tracker_link(m->cfg.task, s->solver);
  MbLaunch<T> L;
  memset(&L.ua, 0, sizeof L.ua);
  memset(&L.pa, 0, sizeof L.pa);
  L.ctx = ctx; L.m = m; L.d = d; L.s = s; L.mult = nullptr; L.Scache = buf.p; L.s_stride = s_stride; L.partial = 1; L.fused_exchange = false;
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int rows = (int)std::min<int64_t>(chunk, n - r0);
    L.row_begin = r0; L.rows = rows; L.phase = 0;
    dispatch_layout<T>(m->kp, L);
    comm_allreduce_sum(ctx, buf.p, (size_t)rows * s_stride, sizeof(T) == 8);
    FMWR_LAUNCH(ctx, mb_score_kernel<T>, ceil_div(rows, 8), 256, 0, (const double*)m->scal.p, m->kp, m->cfg.keep_w0, rows, buf.p, s_stride, link,
                (double)s->min_target, (double)s->max_target, ctx->pn_table.p, d->pred64.p + r0);
  }
  return evaluate_dev(ctx, d, m->cfg.task, s->metric);
}

// Data whose values are still uploading (fmwr_train) may go to this trainer when nothing reads them before their batch: no
// tracker (its scoring pass reads every row) and no strided or explicit visit order (its rows are gathered up front).
bool minibatch_streams_values(const fmwr_solver_cfg* s)
{
  return s->mode == FMWR_MODE_MINIBATCH && (s->solver == FMWR_SGD || s->solver == FMWR_FTRL || s->solver == FMWR_TDAP) &&
         s->step_size <= 0 && s->random_step <= 1 && !(s->visit_order && s->n_visit > 0);
}

// eval_d: the training data the tracker scores (the full data when d holds the gathered visits); holdout: the held-out sets
template <class T>
static void train_minibatch_t(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* holdout,
                              fmwr_data* eval_d = nullptr)
{
  FMWR_REQUIRE(s->batch_size > 0, FMWR_ERR_ARG, "batch_size must be positive in minibatch mode");
  if (!eval_d) eval_d = d;
  if (s->random_step > 1 || (s->visit_order && s->n_visit > 0)) {
    // strided / explicit visit sequence (reference random_select, src/util/Random.h:126-132): the visited rows are gathered, in
    // visit order, into a dataset of their own and the batches are consecutive visits; the tracker still scores the full data
    FMWR_REQUIRE(!(ctx->nccl_comm && ctx->world > 1), FMWR_ERR_UNSUPPORTED, "random_step > 1 is not available on a feature-sharded model");
    std::vector<uint32_t> order = visit_order_host(d, s);
    if ((int64_t)order.size() > (int64_t)s->max_iter) order.resize(s->max_iter);
    if (order.empty()) return;
    DBuf<uint32_t> order_dev;
    order_dev.alloc(order.size());
    FMWR_CUDA(cudaMemcpyAsync(order_dev.p, order.data(), 4 * order.size(), cudaMemcpyHostToDevice, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    std::unique_ptr<fmwr_data> visited(data_gather_rows(d, order_dev.p, (int64_t)order.size()));
    fmwr_solver_cfg s2 = *s;
    s2.random_step = 1; s2.visit_order = nullptr; s2.n_visit = 0;
    s2.compat &= ~FMWR_COMPAT_SKIP_ROW0;                   // the sequence already says which rows are visited
    s2.max_iter = (int32_t)order.size();
    train_minibatch_t<T>(ctx, m, visited.get(), &s2, tr, holdout, eval_d);
    return;
  }
  const SolverParams<double> spd = make_params<double>(m, s);
  const bool kept_state = model_alloc_state(m, solver_state_count(spd), s->solver, s->warm_state != 0);

  const int64_t row0 = (s->compat & FMWR_COMPAT_SKIP_ROW0) ? 1 : 0;     // F5: the reference scan starts at row 1
  const int64_t B = s->batch_size;
  const int64_t epoch_rows = d->n - row0;
  if (epoch_rows <= 0) return;
  minibatch_build(d, row0, B);
  const int64_t n_batches = ceil_div64(epoch_rows, B);

  // single GPU: S cache rows are kp wide.  Feature-parallel: kp + 4 (S_f, the additive scalar, padding to keep 16-byte rows)
  const bool multi = ctx->nccl_comm != nullptr && ctx->world > 1;
  const int s_stride = multi ? m->kp + 4 : m->kp;
  // peer window open: the exchange runs inside our own kernels (NVLink stores + flags), no NCCL call per batch
  const bool peer = multi && ctx->peer.ready;
  PeerArgs pa;
  memset(&pa, 0, sizeof pa);
  DBuf<T> mult, Scache;
  if (peer) {
    pa.rank = ctx->rank; pa.world = ctx->world;
    pa.rows_per_owner = (int)ceil_div64(B, ctx->world);
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    pa.off_P = PEER_CTL_BYTES;
    pa.off_S = up(pa.off_P + (size_t)ctx->world * pa.rows_per_owner * s_stride * sizeof(T));
    pa.off_mult = up(pa.off_S + (size_t)B * s_stride * sizeof(T));
    pa.off_msum = up(pa.off_mult + (size_t)B * sizeof(T));
    FMWR_REQUIRE(pa.off_msum + 8192 <= ctx->peer.bytes, FMWR_ERR_COMM,
                 "peer window too small for this batch size / factor count (see fmwr_comm_peer_bytes)");
    for (int r = 0; r < ctx->world; ++r) pa.base[r] = (char*)ctx->peer.base[r];
  }
  mult.alloc(peer ? 1 : B);
  FMWR_REQUIRE((uint64_t)B * (uint64_t)s_stride < (1ull << 32), FMWR_ERR_UNSUPPORTED, "batch_size x factors too large (the S cache is indexed with 32 bits)");
  Scache.alloc(peer ? 1 : (size_t)B * s_stride);
  if (multi && !peer) FMWR_CUDA(cudaMemsetAsync(Scache.p, 0, Scache.bytes(), ctx->stream));
  T* sc_p = peer ? reinterpret_cast<T*>(pa.base[pa.rank] + pa.off_S) : Scache.p;
  T* mult_p = peer ? sc_p + m->kp : mult.p;          // peer mode: the multiplier travels in the padding of the S-cache row

  MbLaunch<T> L;
  L.ctx = ctx; L.m = m; L.d = d; L.s = s; L.mult = mult_p; L.Scache = sc_p; L.s_stride = s_stride; L.partial = peer ? 2 : (multi ? 1 : 0);
  L.pa = pa;
  MbUpdArgs<T>& ua = L.ua;
  memset(&ua, 0, sizeof ua);
  ua.seg_ptr = d->mb_seg_ptr.p; ua.seg_rec = d->mb_seg_rec.p; ua.ent_row = d->mb_ent_row.p; ua.ent_val = d->mb_ent_val.p;
  ua.mult = mult_p; ua.Scache = sc_p;
  ua.peer = peer ? 1 : 0; ua.pa = pa; ua.mult_stride = peer ? s_stride : 1;
  // fp32 models with 32-float rows on long rows: the stream forward kernel runs the exchange itself
  const bool fused_exchange = peer && sizeof(T) == 4 && stream_forward_ok(m, d->nnz, d->n, 2);
  if (fused_exchange) { ua.msum = reinterpret_cast<const double*>(pa.base[pa.rank] + pa.off_msum); ua.msum_n = ctx->world; }
  else if (peer) ua.mult_compact = reinterpret_cast<const T*>(pa.base[pa.rank] + pa.off_mult);
  L.fused_exchange = fused_exchange;
  ua.w = (T*)m->w.p; ua.v = (T*)m->v.p; ua.scal = (double*)m->scal.p;
  for (int i = 0; i < 4; ++i) { ua.sw[i] = (T*)m->sw[i].p; ua.sv[i] = (T*)m->sv[i].p; }
  ua.kp = m->kp; ua.k0 = m->cfg.keep_w0; ua.k1 = m->cfg.keep_w1; ua.s_stride = s_stride;
  ua.sp = make_params<T>(m, s);

  const int64_t max_iter = s->max_iter;
  Tracker trk(ctx, m, s, tr, holdout);
  int64_t iter = 0;
  bool stop = false;
  double u_w = 0.0, u_v = 0.0;
  const bool sgd_l1 = spd.solver == FMWR_SGD && spd.l1;
  if (sgd_l1 && kept_state) {                // cumulative-L1 totals live in the scalar block ([1], [2]) like in the exact mode
    double h[2] = {0, 0};
    FMWR_CUDA(cudaMemcpyAsync(h, (double*)m->scal.p + 1, 16, cudaMemcpyDeviceToHost, ctx->stream));
    FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
    u_w = h[0]; u_v = h[1];
  }
  // The per-batch launches are recorded into CUDA graphs (chunks of GRAPH_CHUNK batches) and replayed by the device,
  // so the epoch does not depend on host launch latency / host jitter.  Per-kernel profiling, the tracker and the
  // NCCL path use plain launches.
  // one-shot path: the values of batch b may still be crossing PCIe; each batch waits for its chunk and fills its CSC values
  const bool pending0 = d->mb_vals_pending;
  const bool use_graph = !ctx->profile && trk.step <= 0 && (!multi || peer) && !pending0 && getenv("FMWR_NO_GRAPH") == nullptr;
  constexpr int GRAPH_CHUNK = 2048;
  // owns the graphs; if anything throws while the stream is capturing, the destructor ends and abandons the capture so the
  // context's stream stays usable for the next call
  struct GraphBag {
    cudaStream_t stream; bool capturing = false;
    std::vector<cudaGraphExec_t> execs; std::vector<cudaGraph_t> graphs;
    ~GraphBag()
    {
      if (capturing) { cudaGraph_t g = nullptr; cudaStreamEndCapture(stream, &g); if (g) cudaGraphDestroy(g); cudaGetLastError(); }
      for (auto ge : execs) cudaGraphExecDestroy(ge);
      for (auto g : graphs) cudaGraphDestroy(g);
    }
  } bag;
  bag.stream = ctx->stream;
  int captured = 0;
  auto flush_graph = [&]() {
    if (!use_graph || captured == 0) return;
    cudaGraph_t g = nullptr;
    bag.capturing = false;
    FMWR_CUDA(cudaStreamEndCapture(ctx->stream, &g));
    bag.graphs.push_back(g);
    cudaGraphExec_t ge = nullptr;
    FMWR_CUDA(cudaGraphInstantiate(&ge, g, 0));
    bag.execs.push_back(ge);
    FMWR_CUDA(cudaGraphLaunch(ge, ctx->stream));
    captured = 0;
  };
  while (iter < max_iter && !stop) {
    for (int64_t b = 0; b < n_batches && iter < max_iter; ++b) {
      if (use_graph && captured == 0) { FMWR_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal)); bag.capturing = true; }
      const int64_t rb = row0 + b * B;
      minibatch_batch_values(d, b);
      int64_t rows = std::min<int64_t>(B, d->n - rb);
      rows = std::min<int64_t>(rows, max_iter - iter);
      L.row_begin = rb; L.rows = (int)rows;
      L.phase = 0;
      dispatch_layout<T>(m->kp, L);
      if (peer && !fused_exchange) {
        L.phase = 2;
        dispatch_layout<T>(m->kp, L);
      } else if (peer) {
        // the stream forward kernel did the owner's reduction itself (forward_stream.cuh)
      } else if (multi) {
        // one exchange per minibatch: sum the per-row partials over the feature shards (NCCL over NVLink / NVSwitch)
        comm_allreduce_sum(ctx, Scache.p, (size_t)rows * s_stride, sizeof(T) == 8);
        FMWR_LAUNCH(ctx, mb_finalize_kernel<T>, ceil_div(rows, 8), 256, 0, d->y.p, (const double*)m->scal.p, m->kp, m->cfg.keep_w0,
                    m->cfg.task, T(s->min_target), T(s->max_target), rb, (int)rows, Scache.p, s_stride, mult.p);
      }
      if (spd.solver == FMWR_SGD && spd.l1) { u_w += (double)rows * spd.lr * spd.reg_w; u_v += (double)rows * spd.lr * spd.reg_v; }
      ua.seg_begin = (uint32_t)d->mb_batch_seg[b]; ua.seg_end = (uint32_t)d->mb_batch_seg[b + 1];
      ua.row_begin = rb; ua.rows = (int)rows; ua.u_w = T(u_w); ua.u_v = T(u_v);
      L.phase = 1;
      dispatch_layout<T>(m->kp, L);
      iter += rows;
      if (use_graph && ++captured >= GRAPH_CHUNK) flush_graph();
      if (trk.due_after_batch(iter)) {
        const double score = multi ? tracker_score_sharded<T>(ctx, m, eval_d, s) : tracker_score(ctx, m, eval_d, s);
        stop = trk.record(iter - 1, score);
        if (stop) break;
      }
    }
  }
  minibatch_all_values(d);                       // a truncated first epoch: finish the value fill for later calls
  flush_graph();
  if (sgd_l1) { const double h[2] = {u_w, u_v}; FMWR_CUDA(cudaMemcpyAsync((double*)m->scal.p + 1, h, 16, cudaMemcpyHostToDevice, ctx->stream)); }
  trk.restore_best();
  FMWR_CUDA(cudaStreamSynchronize(ctx->stream));
  if (peer) peer_check_error(ctx);
  if (peer && getenv("FMWR_PEER_DEBUG")) {
    unsigned long long h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    void* dp = reinterpret_cast<uint32_t*>(pa.base[pa.rank]) + PEER_DEBUG;
    FMWR_CUDA(cudaMemcpy(h, dp, sizeof h, cudaMemcpyDeviceToHost));
    FMWR_CUDA(cudaMemset(dp, 0, sizeof h));
    if (h[3]) fprintf(stderr, "[fmwr peer] rank %d: per CTA and launch: partial pass %.1f us, first barrier %.1f us, owner reduction %.1f us (%llu CTA-launches)\n",
                      ctx->rank, h[0] / 1e3 / h[3], h[1] / 1e3 / h[3], h[2] / 1e3 / h[3], h[3]);
    if (h[3] && h[6]) fprintf(stderr, "[fmwr peer] rank %d: start -> second arrival %.1f us (avg CTA), start -> flags out %.1f us (last CTA)\n", ctx->rank,
                              h[4] / 1e3 / h[3], h[5] / 1e3 / h[6]);
  }
  trk.write_trace(iter);
}

void train_minibatch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* holdout)
{
  if (m->prec == FMWR_F64) train_minibatch_t<double>(ctx, m, d, s, tr, holdout);
  else train_minibatch_t<float>(ctx, m, d, s, tr, holdout);
}

}  // namespace fmwr
