// Stream forward: the FM forward pass for fp32 models with 29..32 factors (one 128-byte factor row per feature) as a
// software-pipelined walk over the flat CSR entry stream.
//
// team_gather (forward.cuh) fetches a row's factor rows in batches (issue U, consume U) that end at the row's end: with 39
// non-zeros per row the loads in flight per lane swing between U and 0 and every row pays a pipeline fill.  The
// micro-benchmark profiles/tools/gather_bench.cu shows what the memory system gives for this exact access pattern (random
// 128-byte rows from a 128 MB table): 3.85 ms per 390 M rows with 8 loads per lane kept in flight, 5.5 ms with 4.
// Here an 8-lane group owns a CONTIGUOUS range of rows, i.e. a contiguous range of CSR entries, and walks it with a
// rotating register ring of 8 factor-row vectors: as soon as entry t has been consumed its register is re-issued for
// entry t + 8, across row boundaries, so 8 loads per lane stay in flight for the whole launch.  Column ids and values
// arrive as coalesced 8-entry chunks (one per lane, two chunks ahead) and are handed round by shuffles; the linear term is
// gathered once per chunk (lane l owns entry l) and folded in when its entry is consumed.  A row is finalised when the
// walk reaches its end offset: 3-stage group reduction, then the mode's epilogue.
//
// Arithmetic per entry is team_gather's (P_f += t S_f; S_f += t, reference src/core/Model.h:144-158 without the
// cancellation); only the order of the final reduction over lanes differs.
#pragma once
#include "forward.cuh"
#include <algorithm>

namespace fmwr {

constexpr int SF_BLOCKS = 3;     // 78 registers, no spills; at 4 (64 registers) ptxas rematerialises every shared-memory address per step
__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
enum { SF_PREDICT = 0, SF_TRAIN = 1, SF_PARTIAL = 2, SF_PARTIAL_PEER = 3 };

struct SfArgs {
  const uint32_t* rowptr; const uint32_t* col; const float* val; const float* y;
  const float* w; const float* v; const double* scal;
  int k0, k1, task;
  float lo, hi;
  int64_t row_begin; int64_t rows;       // rows [row_begin, row_begin + rows) of the data handle
  int rpg;                                // rows per 8-lane group (stream_grid)
  int debug;                              // SF_PARTIAL_PEER: accumulate the phase timers (FMWR_PEER_DEBUG)
  double* out;                            // SF_PREDICT: raw scores (the link runs as a second, elementwise pass)
  float* mult; float* Scache; int s_stride;   // SF_TRAIN / SF_PARTIAL*: per-row multiplier and S cache (row index relative to row_begin)
  PeerArgs pa;
};

template <int MODE>
__global__ void __launch_bounds__(256, SF_BLOCKS) forward_stream_kernel(SfArgs a)
{
  constexpr int LPR = 8, U = 8;
  const int lane = threadIdx.x & 31, g = lane >> 3, l = lane & 7;
  const unsigned gmask = 0xffu << (g * 8);
  const int gl = g * 8;                                   // first lane of the group
  // rows are counted in 32 bits (a launch covers < 2^31 rows: callers split larger ranges)
  const int group = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 4 + g;
  const int rpg = a.rpg;
  uint32_t ep_base = 0u;
  unsigned long long t_start = 0;
  if (MODE == SF_PARTIAL_PEER && a.debug && threadIdx.x == 0) t_start = globaltimer_ns();
  if (MODE == SF_PARTIAL_PEER)       // EPOCH2 is only bumped after every CTA of the previous launch passed its last barrier: stable here
    ep_base = *reinterpret_cast<volatile uint32_t*>(reinterpret_cast<uint32_t*>(peer_base(a.pa, a.pa.rank)) + PEER_EPOCH2);
  int r = (int)min((int64_t)group * rpg, a.rows);         // current row (relative to row_begin)
  const int r1 = (int)min((int64_t)r + rpg, a.rows);
  if (r < r1) {
    const uint32_t* __restrict__ rp = a.rowptr + a.row_begin;
    const float w0 = a.k0 ? (float)a.scal[0] : 0.f;
    const uint32_t E0 = __ldg(rp + r), E1 = __ldg(rp + r1);
    uint32_t row_end = __ldg(rp + r + 1);
    uint32_t next_end = r + 2 <= r1 ? __ldg(rp + r + 2) : 0xffffffffu;
    const float* __restrict__ vl = a.v + l * 4;

    float S[4] = {0.f, 0.f, 0.f, 0.f}, P[4] = {0.f, 0.f, 0.f, 0.f};
    float pend = 0.f;
    const int r_first = r;

    auto finalize = [&]() {
      float part = (P[0] + P[1]) + (P[2] + P[3]);          // the linear term was folded into P[0]
      if (MODE >= SF_PARTIAL) part -= 0.5f * ((S[0] * S[0] + S[1] * S[1]) + (S[2] * S[2] + S[3] * S[3]));
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) part += __shfl_xor_sync(gmask, part, o);
      if (MODE == SF_PREDICT) {
        // scores are parked one per lane and leave as runs of up to 8 consecutive doubles (two full sectors): a lone 8-byte
        // store per row would hand L2 four partial writes per sector, 39 steps apart
        const int64_t row = a.row_begin + r;
        if (l == (int)(row & 7)) pend = w0 + part;
        if ((row & 7) == 7 || r == r1 - 1) {
          const int64_t rr = (row & ~(int64_t)7) + l;
          if (rr >= a.row_begin + r_first && rr <= row) a.out[rr] = (double)pend;
        }
      } else if (MODE == SF_TRAIN) {
        if (l == 0) a.mult[r] = grad_mult_fast(a.task, w0 + part, __ldg(a.y + a.row_begin + r), a.lo, a.hi);
        reinterpret_cast<float4*>(a.Scache + (size_t)r * a.s_stride)[l] = make_float4(S[0], S[1], S[2], S[3]);
      } else if (MODE == SF_PARTIAL) {
        if (l == 0) a.Scache[(size_t)r * a.s_stride + 32] = part;
        reinterpret_cast<float4*>(a.Scache + (size_t)r * a.s_stride)[l] = make_float4(S[0], S[1], S[2], S[3]);
      } else {
        const int owner = r / a.pa.rows_per_owner;
        float* dst = reinterpret_cast<float*>(peer_base(a.pa, owner) + a.pa.off_P) +
                     ((size_t)a.pa.rank * a.pa.rows_per_owner + (size_t)(r - owner * a.pa.rows_per_owner)) * a.s_stride;
        if (l == 0) *reinterpret_cast<float4*>(dst + 32) = make_float4(part, 0.f, 0.f, 0.f);     // whole 16-byte vector: no partial sector over NVLink
        reinterpret_cast<float4*>(dst)[l] = make_float4(S[0], S[1], S[2], S[3]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) { S[i] = 0.f; P[i] = 0.f; }
      ++r;
      row_end = next_end;
      next_end = r + 2 <= r1 ? __ldg(rp + r + 2) : 0xffffffffu;
    };

    // chunk = 8 consecutive entries, one per lane.  The (column, value) chunks travel global -> shared memory by cp.async, two
    // chunks ahead, into a 4-slot ring per group: no register holds them while they are in flight (a register would have to be
    // parked across the 8 ring steps, and ptxas parks it in local memory right behind the load -- a full-latency stall per chunk)
    __shared__ uint32_t s_col[8][4][4][8];
    __shared__ float s_val[8][4][4][8];
    uint32_t* sc = &s_col[threadIdx.x >> 5][g][0][0];
    float* sx = &s_val[threadIdx.x >> 5][g][0][0];
    auto issue_chunk = [&](uint32_t base, int slot) {
      const uint32_t j = base + l;
      if (j < E1) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(sc + slot * 8 + l)), "l"(a.col + j) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(sx + slot * 8 + l)), "l"(a.val + j) : "memory");
      } else { sc[slot * 8 + l] = 0u; sx[slot * 8 + l] = 0.f; }      // past the range: factor row 0 times 0
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto chunks_landed = [&]() { asm volatile("cp.async.wait_group 0;" ::: "memory"); __syncwarp(gmask); };
    auto lin_of = [&](uint32_t base, int slot) -> float {
      return (a.k1 && base + l < E1) ? __ldg(a.w + sc[slot * 8 + l]) * sx[slot * 8 + l] : 0.f;
    };
    issue_chunk(E0, 0);
    issue_chunk(E0 + 8, 1);
    chunks_landed();
    float4 ring[U];
#pragma unroll
    for (int s = 0; s < U; ++s) ring[s] = ld_nc_v16(reinterpret_cast<const float4*>(vl + (size_t)sc[s] * 32));
    float wl_cur = lin_of(E0, 0), wl_nxt;
    int q = 0;
    for (uint32_t Tc = E0; Tc < E1; Tc += 8, ++q) {
      chunks_landed();                                     // chunk q + 1 (issued one iteration ago) is in shared memory
      issue_chunk(Tc + 16, (q + 2) & 3);
      const int cur = (q & 3) * 8, nxt = ((q + 1) & 3) * 8;
      wl_nxt = lin_of(Tc + 8, (q + 1) & 3);
#pragma unroll
      for (int s = 0; s < U; ++s) {
        const uint32_t te = Tc + s;
        while (r < r1 && te == row_end) finalize();       // every row that ends before entry te (empty rows included)
        const float x = sx[cur + s];                       // 0 past the end of the range: no effect
        {
          const float4 v4 = ring[s];
          float t;
          t = v4.x * x; P[0] = fmaf(t, S[0], P[0]); S[0] += t;
          t = v4.y * x; P[1] = fmaf(t, S[1], P[1]); S[1] += t;
          t = v4.z * x; P[2] = fmaf(t, S[2], P[2]); S[2] += t;
          t = v4.w * x; P[3] = fmaf(t, S[3], P[3]); S[3] += t;
        }
        if (l == s) P[0] += wl_cur;
        ring[s] = ld_nc_v16(reinterpret_cast<const float4*>(vl + (size_t)sc[nxt + s] * 32));      // entry te + 8 takes the register over
      }
      wl_cur = wl_nxt;
    }
    while (r < r1) finalize();                             // the last row and trailing empty rows
  }
  if (MODE == SF_PARTIAL_PEER) {
    // ---- the exchange, fused: this rank's partials are on their way to the rows' owners; now, as the owner of rows
    // [rank * rpo, ...), wait for everybody's partials, sum them IN RANK ORDER (deterministic), form score and multiplier and
    // store the row [S_f totals, multiplier] into every rank's S cache.  The batch's sum of multipliers (the intercept's
    // gradient) is reduced on the way: per group -> per CTA -> the last CTA -> one double per rank in every window, so the
    // update kernel adds `world` numbers instead of walking 65 536 strided multipliers in one CTA.
    const PeerArgs& pa = a.pa;
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    const uint32_t ep = ep_base + 1u;
    // FMWR_PEER_DEBUG: where a CTA's time goes (ns summed over CTAs and launches): [0] partial pass, [1] first barrier, [2] owner's
    // reduction, [3] CTAs counted
    unsigned long long* dbg = a.debug ? reinterpret_cast<unsigned long long*>(ctl + PEER_DEBUG) : nullptr;
    unsigned long long t1 = 0, t2 = 0;
    if (dbg && threadIdx.x == 0) { t1 = globaltimer_ns(); atomicAdd(dbg + 0, t1 - t_start); atomicAdd(dbg + 3, 1ull); }
    if (peer_arrive_last(pa, PEER_COUNT1)) peer_publish(pa, PEER_FLAG1, PEER_EPOCH1, ep);
    peer_wait_ep(pa, PEER_FLAG1, ep);
    if (dbg && threadIdx.x == 0) { t2 = globaltimer_ns(); atomicAdd(dbg + 1, t2 - t1); }
    const int rpo = pa.rows_per_owner;
    const int r_lo = pa.rank * rpo;
    const int n_local = max(0, (int)min((int64_t)(r_lo + rpo), a.rows) - r_lo);
    const float* P = reinterpret_cast<const float*>(peer_base(pa, pa.rank) + pa.off_P);
    const float w0 = a.k0 ? (float)a.scal[0] : 0.f;
    const int ngroups = gridDim.x * (blockDim.x >> 5) * 4;
    double msum = 0.0;
    for (int rl = group; rl < n_local; rl += ngroups) {
      float S[4] = {0.f, 0.f, 0.f, 0.f};
      float add = 0.f;
      for (int h = 0; h < pa.world; ++h) {
        const float* row = P + ((size_t)h * rpo + rl) * a.s_stride;
        const float4 t = __ldcg(reinterpret_cast<const float4*>(row) + l);
        S[0] += t.x; S[1] += t.y; S[2] += t.z; S[3] += t.w;
        if (l == 0) add += __ldcg(row + 32);
      }
      float acc = add + 0.5f * ((S[0] * S[0] + S[1] * S[1]) + (S[2] * S[2] + S[3] * S[3]));
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) acc += __shfl_xor_sync(gmask, acc, o);
      const int r = r_lo + rl;
      const float m = grad_mult_fast(a.task, w0 + acc, __ldg(a.y + a.row_begin + r), a.lo, a.hi);
#pragma unroll
      for (int h = 0; h < 8; ++h) {
        if (h >= pa.world) break;
        float* dst = reinterpret_cast<float*>(pa.base[h] + pa.off_S) + (size_t)r * a.s_stride;
        reinterpret_cast<float4*>(dst)[l] = make_float4(S[0], S[1], S[2], S[3]);
        if (l == 0) *reinterpret_cast<float4*>(dst + 32) = make_float4(m, 0.f, 0.f, 0.f);
      }
      msum += (double)m;
    }
    if (dbg && threadIdx.x == 0) atomicAdd(dbg + 2, globaltimer_ns() - t2);
    __shared__ double s_msum[32];
    if (l == 0) s_msum[(threadIdx.x >> 5) * 4 + g] = msum;
    __syncthreads();
    double* part = reinterpret_cast<double*>(peer_base(pa, pa.rank) + pa.off_msum) + 8;
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < (int)(blockDim.x >> 5) * 4; ++i) t += s_msum[i];
      part[blockIdx.x] = t;
    }
    const bool last2 = peer_arrive_last(pa, PEER_COUNT2);
    if (dbg && threadIdx.x == 0) atomicAdd(dbg + 4, globaltimer_ns() - t_start);      // [4] kernel start -> second arrival, per CTA
    if (last2) {
      // the CTA that arrived last adds the CTAs' partial sums in a fixed order (deterministic), all threads fetching in parallel
      double t = 0.0;
      for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) t += __ldcg(part + i);
      __shared__ double s_fin[256];
      s_fin[threadIdx.x] = t;
      __syncthreads();
      if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int i = 0; i < (int)blockDim.x; ++i) tot += s_fin[i];
#pragma unroll
        for (int h = 0; h < 8; ++h)
          if (h < pa.world) reinterpret_cast<double*>(pa.base[h] + pa.off_msum)[pa.rank] = tot;
      }
      peer_publish(pa, PEER_FLAG2, PEER_EPOCH2, ep);
      if (dbg && threadIdx.x == 0) { atomicAdd(dbg + 5, globaltimer_ns() - t_start); atomicAdd(dbg + 6, 1ull); }    // [5] start -> flags out (last CTA)
    }
    (void)ctl;
  }
}

// raw score -> link, in place (SF_PREDICT's second pass; fp64 like the reference's predict_prob, src/core/Model.h:163-180)
static __global__ void link_inplace_kernel(double* __restrict__ out, int64_t n, int link, double lo, double hi, const double* __restrict__ pnY)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = apply_link(link, out[i], lo, hi, pnY);
}

// Grid of a stream launch: every resident 8-lane group gets the same number of rows (the last one the remainder), so no
// group idles while others walk one row more: rows per group from the resident group count, CTAs from the groups needed.
inline int stream_grid(const fmwr_ctx* ctx, int64_t rows, int* rpg_out)
{
  const int64_t max_groups = (int64_t)ctx->sm_count * SF_BLOCKS * 32;
  int64_t rpg = std::max<int64_t>(1, (rows + max_groups - 1) / max_groups);
  // Long launches: cap the rows per group and let the grid run in waves.  With one contiguous range per resident group the
  // groups of an SM stream from ~100 different 2 MB pages of the CSR arrays at once (on top of the 64 pages of V) and the
  // 128-entry TLB thrashes: predict over 10M rows took 8.9 ms with 704 rows per group, 5.8 ms with 64 (profiles/r02_summary.md)
  rpg = std::min<int64_t>(rpg, 64);
  const int64_t groups = (rows + rpg - 1) / rpg;
  *rpg_out = (int)rpg;
  return (int)std::max<int64_t>(1, (groups + 31) / 32);
}

// the stream kernels serve fp32 models whose padded row is exactly 32 floats, on data with rows long enough to keep a ring busy
// (min_nnz_per_row: 8 for whole rows; the column slices of a feature-sharded model have 39/N non-zeros per row and still take the
// stream kernel, which then also runs the exchange)
inline bool stream_forward_ok(const fmwr_model* m, int64_t nnz, int64_t n, int min_nnz_per_row = 8)
{
  return m->prec == FMWR_F32 && m->kp == 32 && n > 0 && n < (1ll << 31) && nnz >= (int64_t)min_nnz_per_row * n;
}

}  // namespace fmwr
