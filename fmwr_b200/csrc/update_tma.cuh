// K2, dense variant: the coordinate update of the minibatch trainers with the parameter rows staged by TMA.
//
// Inside a batch the (batch, feature) segments are sorted by feature, so a tile of consecutive segments touches an
// ascending run of parameter rows.  When the batch is large against the field (configs[1]: 65 536 rows over 25 641 ids per
// field -> 92 % of the rows are touched) that run is almost contiguous: the tile's rows of theta and of every optimizer-state
// array are ONE contiguous range each.  This kernel moves those ranges with 1-D bulk copies (cp.async.bulk, completion on an
// mbarrier) into a shared-memory ring, lets the lane groups update them in place in shared memory, and writes the ranges back
// with bulk stores: HBM sees full-line streams in both directions and no warp holds a DRAM round trip in registers.  A
// producer warp runs the ring (loads, write-backs); eight consumer warps run the segment gradient and the coordinate steps of
// coord.cuh on shared memory.  The only global gathers left in the consumers are the S-cache lines of the segment's rows (L2-resident).
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
    USE_STATE = (SOLVER != FMWR_SGD || L1) ? 1 : 0,
    NA = 1 + (USE_STATE ? solver_nst(SOLVER) : 0),                 // theta + state arrays
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

// One segment of a dense tile: the segment gradient and the steps of coord.cuh, as seg_finish (train_minibatch.cu), with the
// entry lists and the parameter rows read from the stage.
template <class T, int LPR, int CH, int SOLVER, bool L1, class G>
__device__ __forceinline__ void seg_dense(const MbUpdArgs<T>& a, unsigned char* __restrict__ stage, const uint32_t* __restrict__ hdr, int j, int l)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int NST = solver_nst(SOLVER);
  constexpr bool USE_STATE = G::USE_STATE != 0;
  constexpr bool FAST = sizeof(T) == 4;
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
    for (int u = 0; u < UE; ++u) seg_grad_entry<SOLVER>(Gw, bsum, Gv, th, me[u], xe[u], se[u]);
  };
  round(std::integral_constant<int, 3>(), 0u);
  for (uint32_t i0 = 3; i0 < len; i0 += 2) round(std::integral_constant<int, 2>(), i0);
  seg_grad_close<SOLVER>(Gv, th, bsum);

  // ---- linear weight (lane 0 of the group): staged read, direct store
  if (a.k1 && l == 0) {
    const T* wst = reinterpret_cast<const T*>(stage + G::OFF_W) + hdr[6] + rl;
    T stw[NST];
#pragma unroll
    for (int k = 0; k < NST; ++k) stw[k] = USE_STATE ? wst[(k + 1) * (G::RMAX + 8)] : T(0);
    a.w[c] = coord_step<T, SOLVER, true, FAST, false>(wst[0], Gw, stw, a.sp, L1, a.u_w);
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) a.sw[k][c] = stw[k];
    }
  }
  // ---- factors: update the staged rows in place
  constexpr int ASTRIDE = G::RMAX * G::ROWB;       // bytes between the same row of two staged arrays
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    unsigned char* pr = prow + ch * LPR * 16;
    T st[NST][VN] = {};
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) vec_to_arr(*reinterpret_cast<const V16*>(pr + (k + 1) * ASTRIDE), st[k]);
    }
    coord_step<T, SOLVER, false, FAST, false>(th[ch], Gv[ch], st, a.sp, L1, a.u_v);
    if (USE_STATE) {
#pragma unroll
      for (int k = 0; k < NST; ++k) *reinterpret_cast<V16*>(pr + (k + 1) * ASTRIDE) = arr_to_vec(st[k]);
    }
    *reinterpret_cast<V16*>(pr) = arr_to_vec(th[ch]);
  }
}

}  // namespace fmwr
