// Exact (batch = 1) mode, pipelined across samples: the same serial semantics as exact_kernel (train_exact.cu) -- every sample
// sees the parameters exactly as the reference's loop would have left them (reference src/solver/SGD_Learner.h:79-178,
// FTRL_Learner.h:64-202, TDAP_Learner.h:79-233) -- with several samples in flight.
//
// What is serial in the reference's loop is less than it looks.  Sample t+1 needs from sample t (i) the intercept w0 and its
// optimizer scalars, always, and (ii) the rows of w / V / their state for the COLUMNS THE TWO SAMPLES SHARE, if any.  The score
// is w0 + rest(t+1), and rest (the 39 gathers, the S_f sums) does not involve w0.  So:
//   * one warp owns one sample from gather to write-back (no CTA barrier inside a sample): it copies the parameter and state
//     vectors of the row's columns into its shared-memory stage with cp.async, forms S_f and rest(t) with shuffles, then takes
//     its turn on the SCALAR CHAIN -- wait for the token of sample t-1, score = w0 + rest, multiplier, w0 step (fp64, as the
//     reference's doubles), pass the token on -- and only then runs the coordinate updates and writes them back.  The chain is
//     the only part that is serial for every sample: ~200 cycles for SGD, ~600 for FTRL / TDAP (fp64 sqrt and divide).
//   * column hazards are tracked exactly like a scoreboard: the pipeline warp walks the visit sequence IN ORDER well ahead of
//     the workers and, per sample, looks every column up in a shared-memory table (column -> last sample that contains it),
//     records that sample as the entry's dependency, and enters the sample itself.  A worker may gather only when the samples
//     its entries depend on have published their write-back (a done tag per ring slot).  Read-after-write, write-after-write
//     and write-after-read all reduce to "same column => the later sample waits for the earlier one to finish".  The table is
//     2-way set-associative (4096 sets of 16 bytes: two columns, their last samples and the latest sample EVICTED from the set,
//     all as 16-bit sample numbers -- only distances below the ring depth matter, older samples have finished by construction);
//     a lookup answers with the hit way's sample AND the evicted one, so it can report a dependency too many, never miss one.
// With no shared columns (uniform synthetic data: 0.15 % of neighbouring samples) `teams` samples overlap fully; data whose
// neighbouring rows always share a column degrades to the serial order, one sample at a time, which is what the reference does.
//
// TDAP's z_w[position] quirk (F6, TDAP_Learner.h:207) makes every sample READ the linear state of columns 0 .. nnz-1: a sample
// waits for the last writer of each of those columns like for its own, and a sample that WRITES a column below the longest row
// seen so far waits for every earlier sample (readers are not entered in the table: they do not conflict with each other).
#pragma once

namespace fmwr {

#ifndef XP_RING
#define XP_RING 64       // ring slots: 32 left the fetch warp waiting for free slots (8 samples being fetched, 8 in the hazard warp, 8 in work, 8 written back but unpublished)
#endif
#ifndef XP_RINGN
#define XP_RINGN 48      // ring entries per sample
#endif
#ifndef XP_TEAMS_MAX
#define XP_TEAMS_MAX 12
#endif
constexpr int XP_MAXT = XP_TEAMS_MAX;                 // worker warps = samples in flight
constexpr int XP_R = XP_RING;                   // ring slots (samples staged ahead by the pipeline warp)
constexpr int XP_RN = XP_RINGN;                  // ring entries per sample; longer rows read the rest from global memory
#ifndef XP_BATCH
#define XP_BATCH 8
#endif
constexpr int XP_G = XP_BATCH;                    // samples per pipeline batch
#ifndef XP_NAP
#define XP_NAP 0         // ns between polls of a ring / done tag.  0: plain spinning -- __nanosleep(20) wakes late enough to cost
                         // 50 % on SGD and configs[0] (1.90 vs 1.28, 1.16 vs 0.73 us per sample); the pollers are single instructions
#endif
#ifndef XP_NAP_TOK
#define XP_NAP_TOK 0     // ... of the scalar chain's token (latency-critical)
#endif
#ifndef XP_UNROLL_G
#define XP_UNROLL_G 4
#endif
#ifndef XP_UNROLL_F
#define XP_UNROLL_F 4
#endif
#ifndef XP_UNROLL_U
#define XP_UNROLL_U 2
#endif
#define XP_PRAGMA(x) _Pragma(#x)
#define XP_UNROLL(n) XP_PRAGMA(unroll n)
#ifndef XP_HASH_BITS
#define XP_HASH_BITS 12
#endif
constexpr int XP_LOGH = XP_HASH_BITS, XP_H = 1 << XP_LOGH;      // sets of the hazard table

__device__ __forceinline__ void xp_cp16(void* dst, const void* src)
{
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
template <int BYTES>
__device__ __forceinline__ void xp_cp_word(void* dst, const void* src)
{
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void xp_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void xp_cp_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ uint32_t xp_hash(uint32_t c) { return (c * 2654435761u) >> (32 - XP_LOGH); }
__device__ __forceinline__ uint32_t xp_ld(const volatile uint32_t* p) { return *p; }
// Watchdog of the pollers: every wait in this kernel is for a strictly EARLIER sample (or for the warp that feeds the ring), so
// none can last; if one does (a bug), the kernel traps -- the host sees a CUDA error ("unspecified launch failure") instead of a
// hung GPU.
#ifndef XP_WATCHDOG_CYCLES
#define XP_WATCHDOG_CYCLES 6000000000ll      // ~3 s at 2 GHz; a wait is microseconds
#endif
struct XpSpin {
  uint32_t n = 0; long long t0 = 0;
  __device__ __forceinline__ void tick(const char*, uint32_t)
  {
    if (XP_NAP) __nanosleep(XP_NAP);
    if ((++n & 0xffffu) != 0u) return;
    const long long now = clock64();
    if (t0 == 0) { t0 = now; return; }
    if (now - t0 > XP_WATCHDOG_CYCLES) __trap();       // (no printf: its stack frame cost the FTRL kernel 18 %)
  }
};
// Every thread of this kernel is in ONE CTA, so CTA scope is the widest scope any synchronisation here needs.  __threadfence() /
// __threadfence_block() are fence.sc (MEMBAR.SC.*: 3000-6000 cycles each where measured, profiles/r02_summary.md); the
// acquire-release form orders the same accesses without the sequential-consistency round trip.
__device__ __forceinline__ void xp_fence() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }
// Hand-offs that live entirely in shared memory (ring, tags, the scalar chain) are written and read in program order by one
// warp each: a warp's shared-memory accesses are performed in order, so those only need the compiler kept from moving them.
// The hardware fence (MEMBAR.ALL.CTA, ~1000+ cycles with stores in flight) is kept for what crosses warps through GLOBAL memory:
// a sample's write-back before its done tag, and the gather of a sample that actually waited for one.
__device__ __forceinline__ void xp_order() { asm volatile("" ::: "memory"); }

// hazard table arithmetic on 16-bit sample numbers
__device__ __forceinline__ uint32_t xp_dist(uint32_t q16, uint32_t x16) { return (q16 - x16) & 0xffffu; }
__device__ __forceinline__ uint32_t xp_clip(uint32_t d) { return d < (uint32_t)XP_R ? d : 0u; }     // samples XP_R back have finished: no dependency
// distances (hit way, evicted) of column c in set s; 0 = nothing in flight
__device__ __forceinline__ uint32_t xp_lookup(const uint4 s, uint32_t c, uint32_t q16)
{
  uint32_t dh = 0u;
  if (s.x == c) dh = xp_clip(xp_dist(q16, s.z & 0xffffu));
  else if (s.y == c) dh = xp_clip(xp_dist(q16, s.z >> 16));
  return dh | (xp_clip(xp_dist(q16, s.w & 0xffffu)) << 8);
}
#ifdef XP_OLD_INSERT
__device__ __forceinline__ uint4 xp_insert(uint4 s, uint32_t c, uint32_t q16)
{
  if (s.x == c) { s.z = (s.z & 0xffff0000u) | q16; return s; }
  if (s.y == c) { s.z = (s.z & 0x0000ffffu) | (q16 << 16); return s; }
  const uint32_t d0 = s.x == 0xffffffffu ? 0x10000u : xp_dist(q16, s.z & 0xffffu);
  const uint32_t d1 = s.y == 0xffffffffu ? 0x10001u : xp_dist(q16, s.z >> 16);
  const bool v1 = d1 > d0;                   // the victim: an empty way, else the older one
  const uint32_t vd = v1 ? d1 : d0;
  if (vd < 0x10000u && vd < xp_dist(q16, s.w & 0xffffu)) s.w = v1 ? (s.z >> 16) : (s.z & 0xffffu);      // remember the evicted sample if it is the closest
  if (v1) { s.y = c; s.z = (s.z & 0x0000ffffu) | (q16 << 16); }
  else { s.x = c; s.z = (s.z & 0xffff0000u) | q16; }
  return s;
}
__device__ __forceinline__ bool xp_present(const uint4 s, uint32_t c, uint32_t q16)
{
  return (s.x == c && (s.z & 0xffffu) == q16) || (s.y == c && (s.z >> 16) == q16);
}
#else
// way 0 is the most recently entered column: a new column pushes way 0 to way 1 and what was there out of the set
__device__ __forceinline__ uint4 xp_insert(uint4 s, uint32_t c, uint32_t q16)
{
  if (s.x == c) { s.z = (s.z & 0xffff0000u) | q16; return s; }
  if (s.y != c) { const uint32_t old = s.z >> 16; if (xp_dist(q16, old) < xp_dist(q16, s.w & 0xffffu)) s.w = old; }     // the closest evicted sample is the one remembered
  s.y = s.x; s.x = c; s.z = (s.z << 16) | q16;
  return s;
}
__device__ __forceinline__ bool xp_present(const uint4 s, uint32_t c, uint32_t q16) { return s.x == c && (s.z & 0xffffu) == q16; }
#endif

// shared-memory plan (dynamic): fixed part, then the per-warp stages
struct XpPlan {
  int teams, ecap, na;                     // worker warps, staged entries per sample, staged arrays (theta + state in use)
  size_t off_stage, stage_bytes_per_team, total;
};

struct XpFixed {
  uint32_t fetched[XP_R], loaded[XP_R], done[XP_R];       // tags: relative sample index + 1 (ring filled / hazards known / written back)
  uint32_t mN[XP_R], mB[XP_R], mAll[XP_R], mDep[XP_R];      // row length, first entry, flags, "some entry has a dependency in flight"
  float mY[XP_R];
  uint32_t rCol[XP_R][XP_RN];
  float rVal[XP_R][XP_RN];
  uint16_t rDep[XP_R][XP_RN];              // per entry: distance to the sample that last held its column | distance to the set's evicted sample << 8 (0: none in flight)
  uint16_t rDep2[XP_R][XP_RN];             // F6 only: the same two distances for the column the entry's POSITION names (read by the refresh)
  uint4 hSet[XP_H];                        // {column way 0, column way 1, last sample way 0 | way 1 << 16, latest evicted sample}
  uint32_t wCol[XP_MAXT][XP_RN];           // chunk columns / values of rows that do not fit the stage in one piece
  float wVal[XP_MAXT][XP_RN];
  double sc[8];
  double sq_acc;
  uint32_t tok;
};

template <class T>
inline XpPlan xp_plan(int lc /* 16-byte vectors per factor row */, int spw, bool has_state, int ns, double avg_nnz)
{
  XpPlan pl;
  pl.na = has_state ? 1 + ns : 1;
  const size_t fixed = (sizeof(XpFixed) + 127) / 128 * 128;
  const size_t budget = (size_t)227 * 1024 - fixed - 1024;
  const size_t bpe = (size_t)pl.na * ((size_t)lc * 16 + sizeof(T));
  int want = (int)std::ceil(avg_nnz) + 1;
  want = (want + spw - 1) / spw * spw;
  if (want > XP_RN) want = XP_RN;
  if (want < spw) want = spw;
  int teams = (int)(budget / (bpe * (size_t)want));
  if (teams > XP_MAXT) teams = XP_MAXT;
  // short samples are bound by the hazard warp and the scalar chain; workers beyond 8 only add pollers there (configs[0]:
  // 0.65 us per sample with 8, 0.69 with 12; configs[1] SGD: 0.93 with 8, 0.84 with 12)
  if (avg_nnz * lc < 128.0 && teams > 8) teams = 8;
  if (teams < 1) teams = 1;
  int ecap = (int)(budget / teams / bpe) / spw * spw;
  if (ecap > XP_RN) ecap = XP_RN / spw * spw;
  pl.teams = teams; pl.ecap = ecap;
  pl.off_stage = fixed;
  pl.stage_bytes_per_team = ((size_t)ecap * bpe + 127) / 128 * 128;
  pl.total = fixed + pl.stage_bytes_per_team * teams;
  return pl;
}

template <class T, int LPR, int CH, int SOLVER>
__global__ void __launch_bounds__((XP_MAXT + 3) * 32, 1) exact_pipe_kernel(ExactArgs<T> a, int teams, int ecap, int na, uint32_t off_stage, uint32_t stage_bytes)
{
  typedef typename Vec<T>::type V16;
  constexpr int VN = Vec<T>::N;
  constexpr int LC = LPR * CH;               // vectors per factor row
  constexpr int SPW = 32 / LPR;              // entries a warp covers per round
  constexpr int NS = solver_nst(SOLVER);
  constexpr bool FAST = sizeof(T) == 4;
  constexpr int LINE = 128 / (int)sizeof(T);
  extern __shared__ __align__(128) unsigned char xp_dyn[];
  XpFixed& F = *reinterpret_cast<XpFixed*>(xp_dyn);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kp = a.kp;
  const SolverParams<T> sp = a.sp;
  const bool sgd_l1 = (SOLVER == FMWR_SGD) && sp.l1;
  const bool has_state = (SOLVER != FMWR_SGD) || sp.l1;
  const bool f6 = SOLVER == FMWR_TDAP && a.tdap_zw_index && a.k1;
  // fp32 models: the w0 state stays fp64 but its one constant divisor becomes a multiplication (intercept_step)
  const double inv_alpha_w = 1.0 / (double)sp.alpha_w;
  const int64_t total64 = a.t_end - a.t_begin;
  if (total64 <= 0) return;
  const uint32_t total = (uint32_t)total64;

  // ---- init
  for (int i = tid; i < XP_H; i += blockDim.x) F.hSet[i] = make_uint4(0xffffffffu, 0xffffffffu, 0x80008000u, 0x8000u);
  if (tid < XP_R) { F.fetched[tid] = 0u; F.loaded[tid] = 0u; F.done[tid] = 0u; }
  if (tid < 8) F.sc[tid] = a.scal[tid];
  if (tid == 0) { F.tok = 0u; F.sq_acc = sqrt(SOLVER == FMWR_FTRL ? a.scal[2] : a.scal[1]); }
  __syncthreads();

  const int64_t period = a.order ? a.order_len : (a.skip_row0 ? a.n - 1 : a.n);

  if (warp == teams) {
    // =========================== fetch warp: visit sequence -> ring ===========================
    // batch j = samples [j*G, j*G + G), lane i < G owns sample j*G + i.  Iteration it: row indices of batch it, row bounds and
    // label of batch it-1, entries of batch it-2 (cp.async into the ring); batch it-3's entries have landed and are handed on.
    const uint32_t n_batches = (total + XP_G - 1) / XP_G;
    uint32_t rowA = 0;
    uint32_t bB = 0, eB = 0; float yB = 0.f;
    int64_t pos = lane < XP_G ? (a.t_begin + (int64_t)lane) % period : 0;       // visit position of this lane's sample in batch `it`
    const int64_t step = (int64_t)XP_G % period;
#ifdef FMWR_EXACT_PROF
    long long pp[4] = {0, 0, 0, 0};
#endif
    for (uint32_t it = 0; it < n_batches + 3; ++it) {
#ifdef FMWR_EXACT_PROF
      long long p0 = clock64();
#define PPROF(i) { const long long c_ = clock64(); pp[i] += c_ - p0; p0 = c_; }
#else
#define PPROF(i)
#endif
      uint32_t rowNew = 0, bNew = 0, eNew = 0; float yNew = 0.f;
      if (it < n_batches && lane < XP_G) {
        const uint32_t q = it * XP_G + lane;
        if (q < total) rowNew = a.order ? a.order[pos] : (uint32_t)(a.skip_row0 ? pos + 1 : pos);
        pos += step; if (pos >= period) pos -= period;
      }
      if (it >= 1 && it - 1 < n_batches && lane < XP_G) {
        const uint32_t q = (it - 1) * XP_G + lane;
        if (q < total) { bNew = a.rowptr[rowA]; eNew = a.rowptr[rowA + 1]; yNew = a.y[rowA]; }
      }
      if (it >= 2 && it - 2 < n_batches) {
        if (lane < XP_G) {
          const uint32_t q = (it - 2) * XP_G + lane;
          if (q < total) {
            const int slot = q & (XP_R - 1);
            if (q >= XP_R) { XpSpin sp_; while (xp_ld(&F.done[slot]) < q - XP_R + 1u) sp_.tick("a free ring slot", q); }      // the slot's previous sample has finished
            const uint32_t nnz = eB - bB;
            F.mN[slot] = nnz; F.mB[slot] = bB; F.mY[slot] = yB; F.mAll[slot] = nnz > (uint32_t)ecap ? 1u : 0u;
          }
        }
        __syncwarp();
#pragma unroll 4
        for (int k2 = 0; k2 < 2 * XP_G; ++k2) {
          const uint32_t q = (it - 2) * XP_G + (k2 >> 1);
          if (q >= total) break;
          const int slot = q & (XP_R - 1);
          const uint32_t j = (k2 & 1) * 32 + lane;
          const uint32_t nnz = F.mN[slot], b = F.mB[slot];
          if (j < min(nnz, (uint32_t)XP_RN)) {
            xp_cp_word<4>(&F.rCol[slot][j], a.col + b + j);
            xp_cp_word<4>(&F.rVal[slot][j], a.val + b + j);
          }
        }
      }
      xp_cp_commit();
      PPROF(0)
      asm volatile("cp.async.wait_group 1;" ::: "memory");       // everything but the group just committed: batch it-3 is in
      __syncwarp();
      if (it >= 3 && it - 3 < n_batches) {
        xp_order();
        __syncwarp();
        if (lane < XP_G) {
          const uint32_t q = (it - 3) * XP_G + lane;
          if (q < total) *reinterpret_cast<volatile uint32_t*>(&F.fetched[q & (XP_R - 1)]) = q + 1u;
        }
      }
      bB = bNew; eB = eNew; yB = yNew; rowA = rowNew;
      PPROF(1)
    }
#ifdef FMWR_EXACT_PROF
    if (lane == 0) printf("pipe prof fetch warp: issue %lld, wait+publish %lld cycles/batch of %d\n", pp[0] / (n_batches + 3), pp[1] / (n_batches + 3), XP_G);
#endif
  } else if (warp == teams + 1) {
    // =========================== hazard warp: column -> last sample table, in sample order ===========================
    // Per sample one dependent chain, kept as short as it goes: the sets of all the row's columns are read ONCE (both rounds of
    // 32 lanes in flight together), the answer and the updated set are computed from the same registers, written back, and a
    // single re-read tells every lane whether its insertion survived (two lanes of the warp may have written the same set).
    uint32_t max_nnz = 0;                     // longest row so far: the positions any earlier sample may have read (F6)
#ifdef FMWR_EXACT_PROF
    long long pp[4] = {0, 0, 0, 0};
#endif
    for (uint32_t q = 0; q < total; ++q) {
#ifdef FMWR_EXACT_PROF
      long long p0 = clock64();
#endif
      const int slot = q & (XP_R - 1);
      { XpSpin sp_; while (xp_ld(&F.fetched[slot]) != q + 1u) sp_.tick("the fetch warp", q); }
      xp_order();
      PPROF(0)
      const uint32_t nnz = F.mN[slot], b = F.mB[slot];
      const uint32_t nr = min(nnz, (uint32_t)XP_RN);
      const uint32_t q16 = q & 0xffffu;
      const bool in0 = lane < nr, in1 = lane + 32u < nr;
      const uint32_t c0 = in0 ? F.rCol[slot][lane] : 0u, c1 = in1 ? F.rCol[slot][lane + 32] : 0u;
      const uint32_t h0 = xp_hash(c0), h1 = xp_hash(c1);
      uint4 s0 = make_uint4(0u, 0u, 0u, 0u), s1 = s0, p0s = s0, p1s = s0;
      if (in0) s0 = F.hSet[h0];
      if (in1) s1 = F.hSet[h1];
      if (f6) { if (in0) p0s = F.hSet[xp_hash(lane)]; if (in1) p1s = F.hSet[xp_hash(lane + 32u)]; }
      uint32_t dep0 = in0 ? xp_lookup(s0, c0, q16) : 0u, dep1 = in1 ? xp_lookup(s1, c1, q16) : 0u, posdep0 = 0u, posdep1 = 0u;
      if (f6) {
        // the refresh READS the linear state of column j (= the position): wait for whoever wrote it last.  Reads are not
        // entered in the table (every sample reads positions 0 .. nnz-1; readers do not conflict with each other); a sample
        // that WRITES such a column waits for every earlier sample instead (write_low below).  (Folding these into "every
        // sample since the farthest of the four" serialised 60 % of the samples: an old, finished sample named by a set's
        // evicted field turned into a wait for the three samples in flight.)
        posdep0 = in0 ? xp_lookup(p0s, lane, q16) : 0u; posdep1 = in1 ? xp_lookup(p1s, lane + 32u, q16) : 0u;
        if (in0) F.rDep2[slot][lane] = (uint16_t)posdep0;
        if (in1) F.rDep2[slot][lane + 32] = (uint16_t)posdep1;
      }
      if (in0) F.hSet[h0] = xp_insert(s0, c0, q16);
      if (in1) F.hSet[h1] = xp_insert(s1, c1, q16);
      for (uint32_t j = XP_RN + lane; j < nnz; j += 32) { const uint32_t c = a.col[b + j], h = xp_hash(c); F.hSet[h] = xp_insert(F.hSet[h], c, q16); }
      if (in0) F.rDep[slot][lane] = (uint16_t)dep0;
      if (in1) F.rDep[slot][lane + 32] = (uint16_t)dep1;
      { const bool anyd = __any_sync(0xffffffffu, (dep0 | dep1 | posdep0 | posdep1) != 0u); if (lane == 0) F.mDep[slot] = anyd ? 1u : 0u; }
      if (f6) {
        max_nnz = max(max_nnz, nnz);
        bool write_low = (in0 && c0 < max_nnz) || (in1 && c1 < max_nnz);
        for (uint32_t j = XP_RN + lane; j < nnz; j += 32) write_low |= a.col[b + j] < max_nnz;
        if (__any_sync(0xffffffffu, write_low) && lane == 0) F.mAll[slot] |= 2u;      // writes a column some earlier sample's refresh may read
      }
      __syncwarp();
      // an insertion that lost its set to another lane's write is remembered as evicted by this very sample
      if (in0 && !xp_present(F.hSet[h0], c0, q16)) F.hSet[h0].w = q16;
      if (in1 && !xp_present(F.hSet[h1], c1, q16)) F.hSet[h1].w = q16;
      for (uint32_t j = XP_RN + lane; j < nnz; j += 32) { const uint32_t c = a.col[b + j], h = xp_hash(c); if (!xp_present(F.hSet[h], c, q16)) F.hSet[h].w = q16; }
      PPROF(1)
      xp_order();
      __syncwarp();
      if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&F.loaded[slot]) = q + 1u;
      PPROF(2)
    }
#ifdef FMWR_EXACT_PROF
    if (lane == 0) printf("pipe prof hazard warp: wait fetched %lld, table %lld, publish %lld cycles/sample\n", pp[0] / total, pp[1] / total, pp[2] / total);
#endif
  } else if (warp == teams + 2) {
    // =========================== hint warp: L2 prefetch of every parameter / state line of the staged samples ===========================
    for (uint32_t q = 0; q < total; ++q) {
      const int slot = q & (XP_R - 1);
      // a hint for a sample the workers already passed is useless: skip ahead instead of falling behind
      if (xp_ld(&F.done[slot]) >= q + 1u || xp_ld(&F.loaded[slot]) > q + 1u) continue;
      { XpSpin sp_; while (xp_ld(&F.fetched[slot]) < q + 1u) sp_.tick("the fetch warp (hints)", q); }
      __syncwarp();
      xp_order();
      if (xp_ld(&F.fetched[slot]) != q + 1u) continue;         // the slot moved on
      const uint32_t nr = min(F.mN[slot], (uint32_t)XP_RN);
      for (uint32_t j = lane; j < nr; j += 32) {
        const uint32_t c = F.rCol[slot][j];
        const size_t off = (size_t)c * kp;
        for (int x = 0; x < kp; x += LINE) {
          prefetch_l2(a.v + off + x);
          if (has_state) {
#pragma unroll
            for (int s = 0; s < NS; ++s) prefetch_l2(a.sv[s] + off + x);
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
  } else if (warp < teams) {
    // =========================== worker warps: one sample each ===========================
    const int slotw = lane / LPR, l = lane % LPR;
    unsigned char* const stage = xp_dyn + off_stage + (size_t)warp * stage_bytes;
    V16* const stV = reinterpret_cast<V16*>(stage);                                            // [na][ecap * LC]
    T* const stW = reinterpret_cast<T*>(stage + (size_t)na * ecap * LC * sizeof(V16));          // [na][ecap]
    const size_t vstride = (size_t)ecap * LC;
#ifdef FMWR_EXACT_PROF
    long long pt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define XPROF(i) { const long long c_ = clock64(); pt[i] += c_ - p0; p0 = c_; }
#else
#define XPROF(i)
#endif
    uint32_t pending = 0xffffffffu;          // this warp's previous sample: written back, done tag not yet published
    for (uint32_t q = (uint32_t)warp; q < total; q += (uint32_t)teams) {
#ifdef FMWR_EXACT_PROF
      long long p0 = clock64();
#endif
      const int slot = q & (XP_R - 1);
      { XpSpin sp_; while (xp_ld(&F.loaded[slot]) != q + 1u) sp_.tick("the hazard warp", q); }
      XPROF(0)
      __syncwarp();
      xp_order();
      const uint32_t nnz = F.mN[slot], b = F.mB[slot];
      const T yv = T(F.mY[slot]);
      const uint32_t flags = F.mAll[slot];
      const bool chunked = (flags & 1u) != 0u;          // the row does not fit the stage in one piece
      const bool wait_all = flags != 0u;                // ... or writes a column earlier samples read by position (F6): wait for everybody
      // ---- hazards: the samples this one's columns were last seen in must have written back
      // (a dependency whose done tag is already up needs nothing: its write-back was fenced before the tag, long ago)
      auto open_dep = [&](uint32_t dist) -> bool { if (dist == 0u || dist > q) return false; const uint32_t d = q - dist; return xp_ld(&F.done[d & (XP_R - 1)]) < d + 1u; };
      bool has_dep = false;
      if (wait_all) { if (lane >= 1 && lane < teams) has_dep = open_dep((uint32_t)lane); }
#ifdef XP_NO_MDEP
      else {
#else
      else if (F.mDep[slot]) {
#endif
        for (uint32_t j = lane; j < nnz; j += 32) {
          const uint32_t dd = F.rDep[slot][j] | (f6 ? (uint32_t)F.rDep2[slot][j] << 16 : 0u);
          if (dd) has_dep |= open_dep(dd & 0xffu) | open_dep((dd >> 8) & 0xffu) | open_dep((dd >> 16) & 0xffu) | open_dep(dd >> 24);
        }
      }
      has_dep = __any_sync(0xffffffffu, has_dep) && !a.nohazard;      // FMWR_EXACT_NOHAZARD=1: the tests' proof that the tracker matters
      // this warp's previous sample publishes its write-back late (below, once its stores have had a forward pass to land);
      // a sample that is about to wait for others publishes it first: the sample it waits for may be that very one
      if (has_dep && pending != 0xffffffffu) {
        xp_fence();
        __syncwarp();
        if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&F.done[pending & (XP_R - 1)]) = pending + 1u;
        pending = 0xffffffffu;
      }
      if (!has_dep) {
      } else if (wait_all) {
        if (lane >= 1 && lane < teams && q >= (uint32_t)lane) { const uint32_t d = q - lane; XpSpin sp_; while (xp_ld(&F.done[d & (XP_R - 1)]) < d + 1u) sp_.tick("all earlier samples", q); }
      } else {
        for (uint32_t j = lane; j < nnz; j += 32) {
          const uint32_t dd = F.rDep[slot][j] | (f6 ? (uint32_t)F.rDep2[slot][j] << 16 : 0u);
#pragma unroll
          for (int k2 = 0; k2 < 4; ++k2) {
            const uint32_t dist = (dd >> (8 * k2)) & 0xffu;
            if (dist && dist <= q) { const uint32_t d = q - dist; XpSpin sp_; while (xp_ld(&F.done[d & (XP_R - 1)]) < d + 1u) sp_.tick("a dependency", q); }
          }
        }
      }
      __syncwarp();
      if (has_dep) xp_fence(); else xp_order();
      XPROF(1)

      const uint32_t* ccol = chunked ? F.wCol[warp] : F.rCol[slot];
      const float* cval = chunked ? F.wVal[warp] : F.rVal[slot];
      // one chunk of the row: columns/values (chunked rows), then parameter and state vectors into the stage
      auto gather = [&](uint32_t e0, uint32_t cnt) {
        if (chunked) {
          __syncwarp();
          for (uint32_t i = lane; i < cnt; i += 32) { F.wCol[warp][i] = a.col[b + e0 + i]; F.wVal[warp][i] = a.val[b + e0 + i]; }
          __syncwarp();
        }
XP_UNROLL(XP_UNROLL_G)
        for (uint32_t idx = lane; idx < cnt * LC; idx += 32) {
          const uint32_t en = idx / LC, vi = idx % LC;
          const size_t off = (size_t)ccol[en] * kp + (size_t)vi * VN;
          xp_cp16(stV + idx, a.v + off);
          if (has_state) {
#pragma unroll
            for (int s = 0; s < NS; ++s) xp_cp16(stV + (size_t)(1 + s) * vstride + idx, a.sv[s] + off);
          }
        }
        if (a.k1) {
          for (uint32_t i = lane; i < cnt; i += 32) {
            const uint32_t c = ccol[i];
            xp_cp_word<(int)sizeof(T)>(stW + i, a.w + c);
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) xp_cp_word<(int)sizeof(T)>(stW + (size_t)(1 + s) * ecap + i, a.sw[s] + c);
            }
          }
        }
        xp_cp_commit();
        xp_cp_wait_all();
        __syncwarp();
      };

      // ---- forward: S_f, the pairwise correction and the linear term (Model::predict, reference src/core/Model.h:75-103)
      T S[CH][VN];
#pragma unroll
      for (int ch = 0; ch < CH; ++ch)
#pragma unroll
        for (int i = 0; i < VN; ++i) S[ch][i] = T(0);
      T qsum = T(0), lin = T(0);
      for (uint32_t e0 = 0; e0 < nnz; e0 += (uint32_t)ecap) {
        const uint32_t cnt = min((uint32_t)ecap, nnz - e0);
        gather(e0, cnt);
        if (pending != 0xffffffffu) {
          // the previous sample's done tag: its stores were issued a whole gather (a DRAM round trip) ago, so the fence finds
          // them landed; publishing here rather than after the forward pass takes ~1500 cycles off what a dependent sample waits
          xp_fence();
          __syncwarp();
          if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&F.done[pending & (XP_R - 1)]) = pending + 1u;
          pending = 0xffffffffu;
        }
XP_UNROLL(XP_UNROLL_F)
        for (uint32_t en = slotw; en < cnt; en += SPW) {
          const T x = T(cval[en]);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) {
            T arr[VN];
            vec_to_arr(stV[(size_t)en * LC + ch * LPR + l], arr);
#pragma unroll
            for (int i = 0; i < VN; ++i) { const T tt = arr[i] * x; S[ch][i] += tt; qsum += tt * tt; }
          }
        }
        if (a.k1) for (uint32_t i = lane; i < cnt; i += 32) lin += stW[i] * T(cval[i]);
      }
#pragma unroll
      for (int o = LPR; o < 32; o <<= 1)
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
#pragma unroll
          for (int i = 0; i < VN; ++i) S[ch][i] += __shfl_xor_sync(0xffffffffu, S[ch][i], o);
      T acc = T(-0.5) * qsum + lin;
      if (slotw == 0) {
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
#pragma unroll
          for (int i = 0; i < VN; ++i) acc += T(0.5) * S[ch][i] * S[ch][i];
      }
      const T rest = warp_sum(acc);
      if (pending != 0xffffffffu) {            // a row without entries never entered the loop above
        xp_fence();
        __syncwarp();
        if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&F.done[pending & (XP_R - 1)]) = pending + 1u;
        pending = 0xffffffffu;
      }
      XPROF(2)

      // ---- the scalar chain: w0, multiplier, w0's optimizer step, in sample order
      T mult = T(0), u_w = T(0), u_v = T(0);
      if (lane == 0) {
        { XpSpin sp_; while (xp_ld(&F.tok) != q) sp_.tick("the token", q); }
        XPROF(3)
        xp_order();
        volatile double* sc = F.sc;
        double s[6];
        for (int i = 0; i < 6; ++i) s[i] = sc[i];
        const T score = (a.k0 ? T(s[0]) : T(0)) + rest;
        mult = FAST ? grad_mult_fast(a.task, score, yv, T(a.lo), T(a.hi)) : grad_mult<T>(a.task, score, yv, T(a.lo), T(a.hi));
        // cumulative-L1 totals advance once per sample, before the updates (SGD_Learner.h:92-97)
        if (sgd_l1) { s[1] += (double)sp.lr * (double)sp.reg_w; s[2] += (double)sp.lr * (double)sp.reg_v; u_w = T(s[1]); u_v = T(s[2]); }
        double sq_acc = SOLVER == FMWR_SGD ? 0.0 : F.sq_acc;
        intercept_step<T, SOLVER, sizeof(T) == 4>(s, (double)mult, a.k0, sq_acc, sp, inv_alpha_w);
        if (SOLVER != FMWR_SGD && a.k0) F.sq_acc = sq_acc;
        for (int i = 0; i < 6; ++i) sc[i] = s[i];
        xp_order();
        *reinterpret_cast<volatile uint32_t*>(&F.tok) = q + 1u;
      }
      XPROF(4)
      mult = __shfl_sync(0xffffffffu, mult, 0);
      if (sgd_l1) { u_w = __shfl_sync(0xffffffffu, u_w, 0); u_v = __shfl_sync(0xffffffffu, u_v, 0); }

      // ---- coordinate updates with the frozen S_f and multiplier; each (feature, factor) is touched once
      for (uint32_t e0 = 0; e0 < nnz; e0 += (uint32_t)ecap) {
        const uint32_t cnt = min((uint32_t)ecap, nnz - e0);
        if (chunked) gather(e0, cnt);        // rows of one chunk still have their stage from the forward
XP_UNROLL(XP_UNROLL_U)
        for (uint32_t en = slotw; en < cnt; en += SPW) {
          const T x = T(cval[en]);
          const size_t off = (size_t)ccol[en] * kp;
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) {
            const int vi = ch * LPR + l;
            const size_t idx = (size_t)en * LC + vi;
            T th[VN], st[NS][VN] = {};
            vec_to_arr(stV[idx], th);
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) vec_to_arr(stV[(size_t)(1 + s) * vstride + idx], st[s]);
            }
            // element by element, each gradient formed just before its step: the fp64 steps branch, and gradients formed ahead
            // would stay live across those branches (registers)
#pragma unroll
            for (int i = 0; i < VN; ++i) {
              T s[NS];
              for (int k = 0; k < NS; ++k) s[k] = st[k][i];
              th[i] = coord_step<T, SOLVER, false, FAST, FAST>(th[i], mult * fm_grad(S[ch][i], th[i], x), s, sp, sp.l1, u_v);
              for (int k = 0; k < NS; ++k) st[k][i] = s[k];
            }
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) reinterpret_cast<V16*>(a.sv[s] + off)[vi] = arr_to_vec(st[s]);
            }
            reinterpret_cast<V16*>(a.v + off)[vi] = arr_to_vec(th);
          }
        }
        if (a.k1) {
          for (uint32_t i = lane; i < cnt; i += 32) {
            const uint32_t c = ccol[i];
            const T x = T(cval[i]);
            T th = stW[i], st[NS] = {};
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) st[s] = stW[(size_t)(1 + s) * ecap + i];
            }
            if (SOLVER == FMWR_TDAP && a.tdap_zw_index) (void)coord_step<T, SOLVER, true, FAST, FAST>(th, mult * x, st, sp, sp.l1, u_w);   // w: F6 below
            else th = coord_step<T, SOLVER, true, FAST, FAST>(th, mult * x, st, sp, sp.l1, u_w);
            if (has_state) {
#pragma unroll
              for (int s = 0; s < NS; ++s) a.sw[s][c] = st[s];
            }
            if (!(SOLVER == FMWR_TDAP && a.tdap_zw_index)) a.w[c] = th;
          }
        }
      }
      // F6: the linear refresh reads z_w[position in row] (TDAP_Learner.h:207); the state of this sample's columns was stored by
      // this warp just above
      if (f6) {
        __syncwarp();
        for (uint32_t i = lane; i < nnz; i += 32) {
          const uint32_t c = (!chunked) ? ccol[i] : a.col[b + i];
          const T z = a.sw[1][i] - a.sw[3][i];
          a.w[c] = tdap_refresh<T, FAST>(z, a.sw[2][c], sp.l1_w, sp.l2_w);
        }
      }
      XPROF(5)
      pending = q;
      XPROF(6)
    }
    if (pending != 0xffffffffu) {
      xp_fence();
      __syncwarp();
      if (lane == 0) *reinterpret_cast<volatile uint32_t*>(&F.done[pending & (XP_R - 1)]) = pending + 1u;
    }
#ifdef FMWR_EXACT_PROF
    if (lane == 0 && warp < 2) {
      const long long N = (total + teams - 1) / teams;
      printf("pipe prof worker %d (teams %d, ecap %d): wait-loaded %lld, wait-deps+fence %lld, gather+forward %lld, wait-token %lld, chain %lld, update %lld, fence %lld cycles/sample\n",
             warp, teams, ecap, pt[0] / N, pt[1] / N, pt[2] / N, pt[3] / N, pt[4] / N, pt[5] / N, pt[6] / N);
    }
#endif
  }
  __syncthreads();
  if (tid < 8) a.scal[tid] = F.sc[tid];
}

}  // namespace fmwr
