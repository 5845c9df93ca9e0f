// K2, dense variant: the coordinate update of the minibatch trainers with the parameter rows staged by TMA.
//
// Inside a batch the (batch, feature) segments are sorted by feature, so a tile of consecutive segments touches an
// ascending run of parameter rows.  When the batch is large against the field (configs[1]: 65 536 rows over 25 641 ids per
// field -> 92 % of the rows are touched) that run is almost contiguous: the tile's rows of theta and of every optimizer-state
// array are ONE contiguous range each.  This kernel moves those ranges with 1-D bulk copies (cp.async.bulk, completion on an
// mbarrier) into a shared-memory ring, lets the lane groups update them in place in shared memory, and writes the ranges back
// with bulk stores: HBM sees full-line streams in both directions and no warp holds a DRAM round trip in registers.  A
// producer warp runs the ring (loads, write-backs); eight consumer warps do the arithmetic of seg_finish (train_minibatch.cu)
// on shared memory.  The only global gathers left in the consumers are the S-cache lines of the segment's rows (L2-resident).
// Tiles whose row range is too wide for a stage (sparse batches, huge fields) fall back to the gather path of the original
// kernel, segment by segment -- results are identical either way (same per-segment arithmetic, same order).
#pragma once
#include "forward.cuh"
#include "coord.cuh"
#include <type_traits>

namespace fmwr {

// ---- raw PTX: mbarrier + 1-D bulk copies (SASS: SYNCS.*, UBLKCP) --------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("{ .reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0]; }" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
  asm volatile("{ .reg .b64 st; mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1; }" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
  uint32_t ok;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(bar), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src, uint32_t bytes, uint64_t policy)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src), "r"(bytes), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// the cache policy of every bulk copy: evict-normal.  Evict-last on theta with evict-first on the state and the lists moved
// K2 by +-1 % (profiles/r02_summary.md).
__device__ __forceinline__ uint64_t l2_policy()
{
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// ---- stage geometry ------------------------------------------------------------------------------------------------
constexpr int TM_CONS_WARPS = 8;
constexpr int TM_THREADS = (TM_CONS_WARPS + 1) * 32;

template <class T, int LPR, int CH, int SOLVER, bool L1, int TS_, int NS_>
struct TmGeom {
  enum {
    TS = TS_, NS = NS_,
    NST = SOLVER == FMWR_SGD ? 1 : (SOLVER == FMWR_FTRL ? 2 : 4),
    USE_STATE = (SOLVER != FMWR_SGD || L1) ? 1 : 0,
    NA = 1 + (USE_STATE ? NST : 0),                 // theta + state arrays
    RMAX = TS + TS / 2 + TS / 4,                    // rows a stage can hold: the tile's feature range may be 1.75x its segment count
    EMAX = 6 * TS,                                  // entries a stage can hold (the first entry of a segment sits in its record too)
    ROWB = LPR * CH * 16,                           // bytes of one parameter row (kp elements)
    OFF_REC = 0,
    OFF_SEGP = OFF_REC + TS * 16,
    OFF_EROW = OFF_SEGP + (TS + 8) * 4,
    OFF_EVAL = OFF_EROW + (EMAX + 8) * 4,
    OFF_W = OFF_EVAL + (EMAX + 8) * 4,
    OFF_PAR = (OFF_W + NA * (RMAX + 8) * (int)sizeof(T) + 127) / 128 * 128,
    STAGE_BYTES = (OFF_PAR + NA * RMAX * ROWB + 127) / 128 * 128,
    HDR_WORDS = 8,
    SMEM_BYTES = NS * STAGE_BYTES + NS * HDR_WORDS * 4 + 3 * NS * 8 + 128
  };
};

// One segment of a dense tile: same arithmetic as seg_finish (train_minibatch.cu), operands from the stage.
template <class T, int LPR, int CH, int SOLVER, bool L1, class G>
__device__ __forceinline__ void seg_dense(const MbUpdArgs<T>& a, unsigned char* __restrict__ stage, const uint32_t* __restrict__ hdr, int j, int l)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NST = G::NST;
  constexpr bool USE_STATE = G::USE_STATE != 0;
  constexpr bool FAST = sizeof(T) == 4;
  constexpr bool ENTRY_FORM = SOLVER == FMWR_TDAP;
  const SolverParams<T>& sp = a.sp;
  const uint4 rec = reinterpret_cast<const uint4*>(stage + G::OFF_REC)[j];
  const uint32_t c = rec.x, len = rec.y;
  const uint32_t rb32 = (uint32_t)a.row_begin, nrows = (uint32_t)a.rows;
  const uint32_t r0 = rec.z - rb32;
  if (!(r0 < nrows)) return;                       // rows ascend inside a segment: nothing of it in the (truncated) batch
  const uint32_t eb = reinterpret_cast<const uint32_t*>(stage + G::OFF_SEGP)[hdr[3] + j];
  const uint32_t eo = hdr[5] + (eb - hdr[4]);      // position of the segment's first entry in the staged entry lists
  const uint32_t* __restrict__ erow = reinterpret_cast<const uint32_t*>(stage + G::OFF_EROW) + eo;
  const float* __restrict__ eval = reinterpret_cast<const float*>(stage + G::OFF_EVAL) + eo;
  const uint32_t rl = c - hdr[1];
  unsigned char* prow = stage + G::OFF_PAR + (size_t)rl * G::ROWB + l * 16;
  const T* sbase = a.Scache + l * VN;

  T th[CH][VN], Gv[CH][VN];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) vec_to_arr(*reinterpret_cast<const V16*>(prow + ch * LPR * 16), th[ch]);
  // The entry lists are in shared memory, so every S-cache address of the segment is known at once: the first round
  // requests entries 0, 1, 2 together (one L2 round trip for the ~70 % of segments with at most 3 entries), later rounds two.
  T Gw = T(0), bsum = T(0);
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
    for (int k2 = 0; k2 < VN; ++k2) Gv[ch][k2] = T(0);
  auto round = [&](auto ue_tag, uint32_t i0) {
    constexpr int UE = decltype(ue_tag)::value;
    T xe[UE], me[UE];
    V16 se[UE][CH];
#pragma unroll
    for (int u = 0; u < UE; ++u) {
      const uint32_t i = i0 + u;
      const bool in = i < len;
      uint32_t rl2 = r0;
      xe[u] = T(__uint_as_float(rec.w));
      if (i > 0) { rl2 = (in ? erow[i] : 0xffffffffu) - rb32; xe[u] = in ? T(eval[i]) : T(0); }
      const bool ok = rl2 < nrows;                 // false for the padding slot and for rows past a truncated batch
      me[u] = ok ? a.mult[rl2 * (uint32_t)a.mult_stride] : T(0);
      const T* sr = sbase + (ok ? rl2 : 0u) * (uint32_t)a.s_stride;
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) se[u][ch] = reinterpret_cast<const V16*>(sr)[ch * LPR];
    }
#pragma unroll
    for (int u = 0; u < UE; ++u) {
      const T mxe = me[u] * xe[u];
      Gw += mxe;
      if (!ENTRY_FORM) bsum += mxe * xe[u];
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        T s[VN];
        vec_to_arr(se[u][ch], s);
#pragma unroll
        for (int k2 = 0; k2 < VN; ++k2) {
          if (ENTRY_FORM) Gv[ch][k2] += me[u] * fm_grad(s[k2], th[ch][k2], xe[u]);
          else Gv[ch][k2] += mxe * s[k2];
        }
      }
    }
  };
  round(std::integral_constant<int, 3>(), 0u);
  for (uint32_t i0 = 3; i0 < len; i0 += 2) round(std::integral_constant<int, 2>(), i0);
  if (!ENTRY_FORM) {
#pragma unroll
    for (int ch = 0; ch < CH; ++ch)
#pragma unroll
      for (int k2 = 0; k2 < VN; ++k2) Gv[ch][k2] = Gv[ch][k2] - th[ch][k2] * bsum;
  }

  // ---- linear weight (lane 0 of the group): staged read, direct store
  if (a.k1 && l == 0) {
    const T* wst = reinterpret_cast<const T*>(stage + G::OFF_W) + hdr[6] + rl;
    T tw = wst[0];
    T stw[NST];
#pragma unroll
    for (int st = 0; st < NST; ++st) stw[st] = USE_STATE ? wst[(st + 1) * (G::RMAX + 8)] : T(0);
    if (SOLVER == FMWR_SGD) {
      T q = stw[0];
      tw = sgd_step(tw, Gw, sp.lr, sp.reg_w, L1 ? 1 : 0, a.u_w, q);
      if (L1) a.sw[0][c] = q;
    } else if (SOLVER == FMWR_FTRL) {
      tw = ftrl_step<T, FAST>(tw, Gw, stw[0], stw[1 % NST], sp.alpha_w, sp.beta_w, sp.l1_w, sp.l2_w);
      a.sw[0][c] = stw[0]; a.sw[1][c] = stw[1 % NST];
    } else {
      const T z = tdap_state<T, FAST>(tw, Gw, stw[0], stw[1 % NST], stw[2 % NST], stw[3 % NST], sp.alpha_w, sp.egamma);
      a.sw[0][c] = stw[0]; a.sw[1][c] = stw[1 % NST]; a.sw[2][c] = stw[2 % NST]; a.sw[3][c] = stw[3 % NST];
      tw = tdap_refresh<T, FAST>(z, stw[2 % NST], sp.l1_w, sp.l2_w);
    }
    a.w[c] = tw;
  }
  // ---- factors: update the staged rows in place
  constexpr int ASTRIDE = G::RMAX * G::ROWB;       // bytes between the same row of two staged arrays
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    unsigned char* pr = prow + ch * LPR * 16;
    if (SOLVER == FMWR_SGD) {
      T q[VN];
      if (L1) vec_to_arr(*reinterpret_cast<const V16*>(pr + ASTRIDE), q);
#pragma unroll
      for (int i = 0; i < VN; ++i) {
        T qq = L1 ? q[i] : T(0);
        th[ch][i] = sgd_step(th[ch][i], Gv[ch][i], sp.lr, sp.reg_v, L1 ? 1 : 0, a.u_v, qq);
        if (L1) q[i] = qq;
      }
      if (L1) *reinterpret_cast<V16*>(pr + ASTRIDE) = arr_to_vec(q);
    } else if (SOLVER == FMWR_FTRL) {
      T z[VN], nn[VN];
      vec_to_arr(*reinterpret_cast<const V16*>(pr + ASTRIDE), z);
      vec_to_arr(*reinterpret_cast<const V16*>(pr + 2 * ASTRIDE), nn);
#pragma unroll
      for (int i = 0; i < VN; ++i) th[ch][i] = ftrl_step<T, FAST>(th[ch][i], Gv[ch][i], z[i], nn[i], sp.alpha_v, sp.beta_v, sp.l1_v, sp.l2_v);
      *reinterpret_cast<V16*>(pr + ASTRIDE) = arr_to_vec(z);
      *reinterpret_cast<V16*>(pr + 2 * ASTRIDE) = arr_to_vec(nn);
    } else {
      T u[VN], nu[VN], dl[VN], h[VN];
      vec_to_arr(*reinterpret_cast<const V16*>(pr + ASTRIDE), u);
      vec_to_arr(*reinterpret_cast<const V16*>(pr + 2 * ASTRIDE), nu);
      vec_to_arr(*reinterpret_cast<const V16*>(pr + 3 * ASTRIDE), dl);
      vec_to_arr(*reinterpret_cast<const V16*>(pr + 4 * ASTRIDE), h);
#pragma unroll
      for (int i = 0; i < VN; ++i) {
        const T z = tdap_state<T, FAST>(th[ch][i], Gv[ch][i], u[i], nu[i], dl[i], h[i], sp.alpha_v, sp.egamma);
        th[ch][i] = tdap_refresh<T, FAST>(z, dl[i], sp.l1_v, sp.l2_v);
      }
      *reinterpret_cast<V16*>(pr + ASTRIDE) = arr_to_vec(u);
      *reinterpret_cast<V16*>(pr + 2 * ASTRIDE) = arr_to_vec(nu);
      *reinterpret_cast<V16*>(pr + 3 * ASTRIDE) = arr_to_vec(dl);
      *reinterpret_cast<V16*>(pr + 4 * ASTRIDE) = arr_to_vec(h);
    }
    *reinterpret_cast<V16*>(pr) = arr_to_vec(th[ch]);
  }
}

}  // namespace fmwr
