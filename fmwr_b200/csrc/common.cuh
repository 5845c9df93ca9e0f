// fmwr_b200 internal header: error plumbing, device buffers, handle structs, warp helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <stdexcept>
#include <memory>
#include <atomic>
#include <thread>

#include "../../include/fmwr_b200.h"

namespace fmwr {

// ---- errors ---------------------------------------------------------------------------------
struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

void set_last_error(const std::string& msg);

#define FMWR_CUDA(expr)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      char _b[512];                                                                              \
      snprintf(_b, sizeof _b, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(_e), __FILE__,   \
               __LINE__, #expr);                                                                 \
      throw ::fmwr::Error(_e == cudaErrorMemoryAllocation ? FMWR_ERR_NOMEM : FMWR_ERR_CUDA, _b); \
    }                                                                                            \
  } while (0)

#define FMWR_REQUIRE(cond, code, msg)              \
  do {                                             \
    if (!(cond)) throw ::fmwr::Error((code), (msg)); \
  } while (0)

// wraps the body of every extern "C" entry point: nothing throws across the ABI
template <class F>
static inline int guarded(F&& f) noexcept
{
  try {
    f();
    return FMWR_OK;
  } catch (const Error& e) {
    set_last_error(e.what());
    return e.code;
  } catch (const std::exception& e) {
    set_last_error(e.what());
    return FMWR_ERR_ARG;
  } catch (...) {
    set_last_error("unknown failure");
    return FMWR_ERR_ARG;
  }
}

// ---- device buffer ----------------------------------------------------------------------------
// Device memory comes from a per-device caching allocator (api.cu): cudaMalloc / cudaFree of multi-GB blocks cost
// tens of ms each and would dominate the one-shot entry points (fmwr_train, fmwr_predict), which build and drop
// several such blocks per call.  Freed blocks are reused by later requests of the same rounded size; fmwr_mem_trim()
// (also run automatically when cudaMalloc fails) returns them to the driver.
void* dev_alloc(size_t bytes);
void dev_free(void* p, size_t bytes);
void dev_trim();

template <class T>
struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  DBuf() {}
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() { release(); }
  void release()
  {
    if (p) dev_free(p, n * sizeof(T));
    p = nullptr;
    n = 0;
  }
  void alloc(size_t count)
  {
    if (count == n && p) return;
    release();
    if (count == 0) count = 1;
    p = (T*)dev_alloc(count * sizeof(T));
    n = count;
  }
  void ensure(size_t count) { if (count > n) alloc(count); }
  void zero(cudaStream_t s) { if (p) FMWR_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  size_t bytes() const { return n * sizeof(T); }
};

// pinned host staging buffer
template <class T>
struct HBuf {
  T* p = nullptr;
  size_t n = 0;
  ~HBuf() { if (p) cudaFreeHost(p); }
  void ensure(size_t count)
  {
    if (count <= n) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    FMWR_CUDA(cudaMallocHost((void**)&p, count * sizeof(T)));
    n = count;
  }
};

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace fmwr

// ---- handles (C structs named in the public header) ------------------------------------------------
struct fmwr_ctx {
  int device = 0;
  int sm_count = 148;
  int smem_optin = 227 * 1024;   // largest dynamic shared memory a CTA may opt in to
  cudaStream_t stream = nullptr;       // compute stream
  cudaStream_t copy_stream = nullptr;  // H2D / D2H staging
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr};
  int64_t launches = 0;
  int64_t h2d_bytes = 0, d2h_bytes = 0;   // bytes the library copied between host and device on behalf of the caller (fmwr_ctx_transfer_bytes)
  // per-kernel CUDA-event profile (bench.py: roofline.achieved is measured live, on this stream)
  bool profile = false;
  struct ProfRec { const char* tag; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  fmwr::DBuf<double> pn_table;   // fast_pnorm Y table   (2862 f64)
  fmwr::DBuf<double> dp_table;   // fast_dpnorm Y table  (40002 f64)
  fmwr::DBuf<char> flush_buf;    // L2 flush scratch
  // feature-parallel communicator (NCCL, resolved at run time; null on a single GPU)
  void* nccl_comm = nullptr;
  int rank = 0, world = 1;
  // peer window (CUDA IPC over NVLink): base[r] = rank r's window mapped into this process (base[rank] = our own)
  struct PeerWin { void* base[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}; size_t bytes = 0; bool ready = false; unsigned als_step = 0; } peer;
  fmwr::DBuf<double> red_scratch;  // reductions
  fmwr::HBuf<double> h_scalar;
  fmwr::HBuf<uint32_t> h_u32;      // pinned landing zone for small device -> host reads (pageable targets serialise with in-flight uploads)
  fmwr::HBuf<float> h_stage[2];    // pinned staging ring of the host-side f64 -> f32 narrowing (data.cu: value uploader); allocated once
};

struct fmwr_data {
  fmwr_ctx* ctx = nullptr;
  int64_t n = 0, p = 0, nnz = 0;
  bool has_labels = false;
  // CSR
  fmwr::DBuf<uint32_t> rowptr;   // [n+1]
  fmwr::DBuf<uint32_t> col;      // [nnz]
  fmwr::DBuf<float> val;         // [nnz]
  fmwr::DBuf<float> val_raw;     // [nnz] pristine values, kept once a z-score pass rewrote `val` (persistent handles: scales / normalize always start from these)
  fmwr::DBuf<float> y;           // [n]
  // CSC twin (rows ascending inside each column)
  bool has_csc = false;
  fmwr::DBuf<uint32_t> colptr;   // [p+1]
  fmwr::DBuf<uint32_t> crow;     // [nnz]
  fmwr::DBuf<float> cval;        // [nnz]
  // coordinate-pass phases: consecutive feature ranges whose members never share a row
  bool has_phases = false;
  std::vector<uint32_t> phase_begin;   // [n_phases+1]
  // per-batch CSC (minibatch mode): entries sorted by (batch, col, row)
  int64_t mb_batch = 0;          // rows per batch the structure was built for (0: none)
  int64_t mb_row0 = 0;           // first row covered
  fmwr::DBuf<uint32_t> mb_seg_ptr;   // [n_seg+1] entry offsets
  fmwr::DBuf<uint4> mb_seg_rec;      // [n_seg] {feature, length, first row, first value bits}
  fmwr::DBuf<uint32_t> mb_ent_row;   // [nnz'] global row index
  fmwr::DBuf<float> mb_ent_val;      // [nnz']
  std::vector<int64_t> mb_batch_seg;  // [n_batches+1] segment offsets per batch (host)
  // The upload (data.cu).  A background thread converts the caller's f64 values chunk by chunk (val_chunk entries) into the
  // context's pinned staging ring and uploads them as f32 -- half the PCIe bytes of the value stream; up_issued = chunks whose copy
  // and event have been queued (an event must be recorded before anybody waits on it), val_ev[c] = chunk c has arrived, val_ready =
  // all of them.  From a page-locked caller buffer every third chunk goes up raw into val64 instead (val_dev[c]) and is narrowed on
  // the device by its first reader.  data_create_f64 waits for all of it unless the values are deferred, and deferred values go only
  // to the minibatch trainer (minibatch_streams_values), which makes each batch's values ready through minibatch_batch_values.
  cudaEvent_t val_ready = nullptr;
  std::vector<cudaEvent_t> val_ev;
  std::vector<char> val_dev;
  int64_t val_waited = 0;              // chunks whose events the compute stream already waits for (per-batch value fill)
  int64_t val_chunk = 0;
  fmwr::DBuf<double> val64;
  bool val_all_narrowed = true;
  std::thread up_thread;
  std::atomic<int64_t> up_issued{0};
  int64_t up_chunks = 0;
  // one-shot training path (values deferred): the column ids cross PCIe in chunks on the copy stream too (col_ev[c] = chunk c of
  // col_chunk entries has arrived), so the per-batch CSC of the first row groups is built while the later ones are still uploading
  // (data.cu: minibatch_build); everything else waits for all of them first (data_wait_cols)
  std::vector<cudaEvent_t> col_ev;
  int64_t col_chunk = 0;
  bool cols_pending = false;           // uploads queued, CSR not validated yet
  // per-batch CSC built while the values were still in flight: ent_val / seg_rec.w of batch b are filled right before
  // batch b trains, as soon as the value chunks covering its rows have arrived (data.cu: minibatch_batch_values)
  bool mb_vals_pending = false;
  fmwr::DBuf<uint32_t> mb_perm;        // sorted position -> original entry (relative to mb_e0)
  uint32_t mb_e0 = 0;
  std::vector<int64_t> mb_batch_ent;   // [n_batches+1] entries before batch b (== offsets into the sorted entry arrays)
  ~fmwr_data()
  {
    if (up_thread.joinable()) up_thread.join();
    if (val_ready) { cudaEventSynchronize(val_ready); cudaEventDestroy(val_ready); }
    for (cudaEvent_t e : val_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : col_ev) cudaEventDestroy(e);
  }
  // ALS/MCMC layouts (phases, row-major / dense copies), built on first use, dropped when the values change
  std::shared_ptr<void> als_cache;
  // last forward result
  int pred_prec = FMWR_F32;
  fmwr::DBuf<float> pred32;      // [n]
  fmwr::DBuf<double> pred64;     // [n]
  fmwr::DBuf<double> contrib64;  // [nnz] per-entry contributions of the last fmwr_contrib_dev (allocated by its first call)
  double min_y = 0, max_y = 0;
  int64_t min_col_nnz = -1;      // smallest non-zero column count (-1: not computed yet); train_als.cu precision policy
};

struct fmwr_model {
  fmwr_ctx* ctx = nullptr;
  fmwr_model_cfg cfg;
  int64_t p = 0;
  int prec = FMWR_F32;
  int k = 0;    // logical factors
  int kp = 0;   // padded row stride (elements): multiple of the 16-byte vector width, power-of-two lanes
  // parameters: w0 is element 0 of `scal`; see layout notes in DESIGN.md
  fmwr::DBuf<char> scal;     // small scalar block: [0]=w0, optimizer scalars follow (f64 each)
  fmwr::DBuf<char> w;        // [p] real
  fmwr::DBuf<char> v;        // [p][kp] real
  // optimizer state, allocated by the trainer on demand (n_state arrays shaped like w / v)
  int n_state = 0;
  int state_solver = 0;      // solver the state arrays belong to (0: none)
  fmwr::DBuf<char> sw[5];    // per-solver state for w
  fmwr::DBuf<char> sv[5];    // per-solver state for V
  size_t esz() const { return prec == FMWR_F64 ? 8 : 4; }
};

namespace fmwr {

// NCCL all-reduces on the context's stream (comm.cu)
void comm_allreduce_sum(fmwr_ctx* ctx, void* buf, size_t count, bool f64);
void comm_allreduce_max_u32(fmwr_ctx* ctx, uint32_t* buf, size_t count);
void comm_allreduce_sum_u32(fmwr_ctx* ctx, uint32_t* buf, size_t count);
void peer_check_error(fmwr_ctx* ctx);   // throws FMWR_ERR_COMM (and clears the flag) when an in-kernel peer barrier timed out

// ---- device helpers ----------------------------------------------------------------------------
#ifdef __CUDACC__
template <class T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- peer window: control block layout (uint32 words) and in-kernel barriers ---------------------------------------
// [FLAG1 + 32 r]  arrival of rank r at barrier 1 (partials stored)      -- written by rank r into EVERY rank's window
// [FLAG2 + 32 r]  arrival of rank r at barrier 2 (row totals stored)
// EPOCH1/2, COUNT1/2, ERR: local words of the owning rank.  Flags sit in separate 128-byte lines.
enum { PEER_FLAG1 = 0, PEER_FLAG2 = 256, PEER_EPOCH1 = 512, PEER_EPOCH2 = 513, PEER_COUNT1 = 514, PEER_COUNT2 = 515, PEER_ERR = 516, PEER_DEBUG = 768 /* 4 x u64 */,
       PEER_CTL_BYTES = 4096 };

struct PeerArgs {
  char* base[8];       // every rank's window
  int rank, world;
  int rows_per_owner;  // rows of a batch a rank finalises: owner(r) = r / rows_per_owner
  size_t off_P, off_S, off_mult;   // byte offsets of the partial slabs [world][rows_per_owner][stride], S cache [B][stride], mult [B]
  size_t off_msum;                 // fused exchange: [0..8) each rank's sum of multipliers (doubles), [8..) this rank's per-CTA partial sums
};

// pa.base[i] with a run-time i, as a chain of selects: indexing a kernel parameter array dynamically makes the compiler copy
// the whole struct to a per-thread stack frame
__device__ __forceinline__ char* peer_base(const PeerArgs& pa, int i)
{
  char* p = pa.base[0];
#pragma unroll
  for (int h = 1; h < 8; ++h) p = (h == i) ? pa.base[h] : p;
  return p;
}

// __threadfence_system() is fence.sc.sys (MEMBAR.SC.SYS); the release / acquire patterns here need no sequential consistency
// between fences, and the acq_rel form is the cheaper instruction (the cta-scope pair measured 3000-6000 vs < 1000 cycles in the
// exact pipeline, profiles/r02_summary.md).
__device__ __forceinline__ void peer_fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// flag stores AFTER one __threadfence_system(): fence + relaxed stores is the release pattern, and it costs one system-scope
// fence per publication instead of one per peer (st.release.sys in a loop over 8 ranks was 8 fences back to back)
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) { asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

// Called by every thread of every CTA at the END of a kernel whose stores the peers will read: the last CTA to get here
// publishes this rank's arrival (a new epoch number) in every rank's window.
__device__ __forceinline__ void peer_signal(const PeerArgs& pa, int flag_base, int epoch_word, int count_word)
{
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    peer_fence_sys();                                   // this CTA's (peer) stores before the count
    const unsigned done = atomicAdd(ctl + count_word, 1u);
    if (done == gridDim.x - 1) {
      ctl[count_word] = 0u;
      const uint32_t ep = ctl[epoch_word] + 1u;
      ctl[epoch_word] = ep;
      peer_fence_sys();
#pragma unroll
      for (int h = 0; h < 8; ++h)
        if (h < pa.world) st_relaxed_sys(reinterpret_cast<uint32_t*>(pa.base[h]) + flag_base + 32 * pa.rank, ep);
    }
  }
}

// Called by every thread at the START of the kernel that reads what the peers stored.  The local epoch word was bumped
// by this rank's own signalling kernel (earlier in the stream), so it names the barrier to wait for.
__device__ __forceinline__ void peer_wait(const PeerArgs& pa, int flag_base, int epoch_word)
{
  if ((int)threadIdx.x < pa.world) {
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    const uint32_t ep = *reinterpret_cast<volatile uint32_t*>(ctl + epoch_word);
    const uint32_t* f = ctl + flag_base + 32 * threadIdx.x;
    const long long t0 = clock64();
    // plain spinning between polls: __nanosleep wakes late
    while ((int32_t)(ld_acquire_sys(f) - ep) < 0) {
      if (clock64() - t0 > 40000000000ll) { ctl[PEER_ERR] = 1u; break; }   // ~20 s: a peer died; the host reports it
    }
  }
  __syncthreads();
}

// Variants for a kernel that runs BOTH sides of a barrier itself (forward_stream.cuh fuses the partial pass and the owner's
// reduction): the epoch to publish / wait for is passed in, because the local epoch word is bumped by this very kernel's last
// CTA and a CTA that reads it "before or after?" would race.
// peer_arrive_last: every thread of every CTA calls it at the end of a phase; returns true in ALL threads of the CTA that arrived
// last (whose threads then see every other CTA's stores); peer_publish: that CTA's thread 0 sends the flags out.
__device__ __forceinline__ bool peer_arrive_last(const PeerArgs& pa, int count_word)
{
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    peer_fence_sys();                                   // this CTA's (local and peer) stores before the count
    const unsigned done = atomicAdd(ctl + count_word, 1u);
    s_last = done == gridDim.x - 1;
    if (s_last) { ctl[count_word] = 0u; asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
  }
  __syncthreads();
  return s_last != 0;
}

__device__ __forceinline__ void peer_publish(const PeerArgs& pa, int flag_base, int epoch_word, uint32_t ep)
{
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    ctl[epoch_word] = ep;
    peer_fence_sys();
#pragma unroll
    for (int h = 0; h < 8; ++h)
      if (h < pa.world) st_relaxed_sys(reinterpret_cast<uint32_t*>(pa.base[h]) + flag_base + 32 * pa.rank, ep);
  }
}

__device__ __forceinline__ void peer_wait_ep(const PeerArgs& pa, int flag_base, uint32_t ep)
{
  if ((int)threadIdx.x < pa.world) {
    uint32_t* ctl = reinterpret_cast<uint32_t*>(peer_base(pa, pa.rank));
    const uint32_t* f = ctl + flag_base + 32 * threadIdx.x;
    const long long t0 = clock64();
    // poll with plain (relaxed, L1-bypassing) loads and acquire ONCE when the flag is there: an acquire at system scope
    // invalidates the SM's L1, and hundreds of CTAs polling that way slow down the CTAs that are still computing
    while ((int32_t)(*reinterpret_cast<const volatile uint32_t*>(f) - ep) < 0) {
      if (clock64() - t0 > 40000000000ll) { ctl[PEER_ERR] = 1u; break; }
    }
    (void)ld_acquire_sys(f);
  }
  __syncthreads();
}

// 16-byte vector views of the parameter rows
template <class T> struct Vec;
template <> struct Vec<float> { typedef float4 type; enum { N = 4 }; };
template <> struct Vec<double> { typedef double2 type; enum { N = 2 }; };

__device__ __forceinline__ void vec_to_arr(const float4& v, float* a) { a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w; }
__device__ __forceinline__ void vec_to_arr(const double2& v, double* a) { a[0] = v.x; a[1] = v.y; }
__device__ __forceinline__ float4 arr_to_vec(const float* a) { return make_float4(a[0], a[1], a[2], a[3]); }
__device__ __forceinline__ double2 arr_to_vec(const double* a) { return make_double2(a[0], a[1]); }

// splitmix64: the counter hash behind the synthetic data and the native RNG (SURVEY section 8d)
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
#endif

// kernel-launch bookkeeping: every launch of OUR kernels goes through this so gpu_launches is a count, not a guess
#define FMWR_LAUNCH(ctx, kernel, grid, block, smem, ...)                                  \
  do {                                                                                    \
    cudaEvent_t _pe1 = nullptr;                                                           \
    if ((ctx)->profile) _pe1 = ::fmwr::prof_begin((ctx), #kernel);                        \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                      \
    if (_pe1) cudaEventRecord(_pe1, (ctx)->stream);                                       \
    (ctx)->launches++;                                                                    \
    FMWR_CUDA(cudaGetLastError());                                                        \
  } while (0)

cudaEvent_t prof_begin(fmwr_ctx* ctx, const char* tag);   // records the start event, returns the stop event

// padded factor stride: k rounded up so a row is LPR 16-byte vectors with LPR a power of two (<= 32 per chunk)
int padded_k(int k, int prec);

// module entry points (implemented across the .cu files)
void build_link_tables(fmwr_ctx* ctx);
void forward_launch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, int link, double lo, double hi);
void contrib_launch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d);   // raw score into pred64, per-entry contributions into contrib64
void transpose_build(fmwr_data* d);
void launch_iota(fmwr_ctx* ctx, uint32_t* a, int64_t n);
// stable LSD radix sort of (key, value) pairs on the low `bits` key bits (sort.cu); val_in == nullptr: values are 0, 1, 2, ...
void sort_pairs_u32(fmwr_ctx* ctx, const uint32_t* key_in, uint32_t* key_out, const uint32_t* val_in, uint32_t* val_out, int64_t n, int bits);
void sort_pairs_u64(fmwr_ctx* ctx, const uint64_t* key_in, uint64_t* key_out, const uint32_t* val_in, uint32_t* val_out, int64_t n, int bits);
void phases_build(fmwr_data* d);
void minibatch_build(fmwr_data* d, int64_t row0, int64_t batch);
void minibatch_batch_values(fmwr_data* d, int64_t b);   // batch b's values ready on the compute stream (per-batch CSC built while they upload)
void minibatch_all_values(fmwr_data* d);                // every value ready (a first epoch that stopped early)
int64_t minibatch_entries(const fmwr_data* d);          // entries of the per-batch CSC
bool minibatch_streams_values(const fmwr_solver_cfg* s);   // train_minibatch may start on data whose values are still uploading
// Held-out tracking (fmwr_train_holdout_dev): at every tracker record, score each eval set (validated by the caller: labelled,
// distinct, not the training data, same feature count) with the record's model; select the best record on eval[0]
struct Holdout {
  fmwr_data* const* eval; int n_eval;
  double* scores; int max_rec;        // scores[i * max_rec + r] for records r < max_rec
  bool select_best;                   // restore the best record's (w0, w, V) into the model at the end
  int patience;                       // > 0: stop after this many records in a row without an improvement on eval[0]
  int32_t* best_rec;                  // out: the first record with the best eval[0] score, -1 if every score was NaN
};
// ---- tracker (tracker.cu): the reference's Tracker (src/core/Tracker.h), shared by the three trainers ----
int tracker_link(int task, int solver);                                                      // the link of the tracker's scores
double tracker_score(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s);   // train metric of m on d
// One training call's records.  The trainer asks due() (after sample idx in exact mode, at the start of sweep idx in ALS/MCMC)
// or due_after_batch() (minibatch mode: one record per step samples crossed, and at the end) and passes the train score to
// record(): snapshot, convergence rule (SGD/FTRL/TDAP, from the third record on), held-out scores, best copy and patience; true
// means stop.  After its loop it calls restore_best() before its final synchronise and write_trace() after it.  m is the model
// the loop trains (the fp64 shadow of an fp32 ALS/MCMC handle), so snapshots, held-out scores and the best copy come from it.
struct Tracker {
  const int step;                     // step_size after Tracker::init's MAX_REC rule; <= 0: no records
  Tracker(fmwr_ctx* ctx, fmwr_model* m, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* h);
  bool due(int64_t idx) const { return step > 0 && (idx % step == 0 || idx == s->max_iter - 1); }
  bool due_after_batch(int64_t iter);
  bool record(int64_t idx, double score);
  void restore_best();                // held-out tracking: best_rec out, and the best record's (w0, w, V) when select_best
  void write_trace(int64_t iters_done);
 private:
  fmwr_ctx* ctx; fmwr_model* m; const fmwr_solver_cfg* s; fmwr_trace* tr; const Holdout* h;
  int n_rec = 0, conv_times = 0, convergent = 0;
  double old_score = 0.0;
  int64_t next_track = 0;             // minibatch mode: the sample count a batch must pass for the next record
  double best = 0.0;                  // held-out tracking: best eval[0] score so far
  int best_rec = -1, since = 0;       // since: records after best_rec
  DBuf<char> best_w, best_v;          // device copy of the best record's w [p] and V [p][kp], the model's own type
  DBuf<double> best_w0;
  bool record_holdout();              // true: patience says stop
};
void train_exact(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* holdout = nullptr);
void train_minibatch(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Holdout* holdout = nullptr);
// SGDA (fmwr_train_sgda_dev, validated by the caller): SGD in exact mode that learns per-group L2 rates on `valid`; lambda_w [G] and
// lambda_v [G][k] in/out
void train_sgda(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, fmwr_data* valid,
                double* lambda_w, double* lambda_v);
// MCMC posterior mean (fmwr_train_posterior_dev): average the predict.FM prediction of draws burn_in+1 .. max_iter on the
// training rows and on every eval set (validated by the caller: distinct, not the training data, same feature count)
struct Posterior {
  int burn_in;
  fmwr_data* const* eval; int n_eval;
};
void train_als_mcmc(fmwr_ctx* ctx, fmwr_model* m, fmwr_data* d, const fmwr_solver_cfg* s, fmwr_trace* tr, const Posterior* post = nullptr,
                    const Holdout* holdout = nullptr);
// shape check of Model::predict_batch (reference src/core/Model.h:112-113)
inline void require_same_features(const fmwr_model* m, const fmwr_data* d)
{
  FMWR_REQUIRE(d->p == m->p, FMWR_ERR_SHAPE, "number of input's features is not correct...");
}
double evaluate_dev(fmwr_ctx* ctx, fmwr_data* d, int task, int metric);
bool model_alloc_state(fmwr_model* m, int n_state, int solver, bool warm);
void model_get_host(fmwr_model* m, double* w0, double* w, double* v);
void model_set_host(fmwr_model* m, double w0, const double* w, const double* v);
double model_get_w0(fmwr_model* m);
void data_scales(fmwr_data* d, const int32_t* norm_cols, int64_t n_norm, double* mean, double* sd);
void data_normalize(fmwr_data* d, const double* mean, const double* sd);
void data_values_from_raw(fmwr_data* d);
void data_restore_values(fmwr_data* d);
void data_set_labels(fmwr_data* d, const double* labels);
void data_synth(fmwr_ctx* ctx, int64_t n, int64_t row_begin, int32_t n_fields, const int64_t* field_size, const int32_t* skew,
                int32_t value_mode, int32_t label_mode, double noise, uint64_t seed, fmwr_data** out);
void model_init_random(fmwr_model* m, double mean, double sd, uint64_t seed);
fmwr_data* data_slice_columns(fmwr_data* src, int64_t c0, int64_t c1);
fmwr_data* data_concat_rows(fmwr_data* const* parts, int n_parts);
fmwr_data* data_gather_rows(fmwr_data* src, const uint32_t* order_dev, int64_t m);
std::vector<uint32_t> visit_order_host(const fmwr_data* d, const fmwr_solver_cfg* s);
void link_table_eval(fmwr_ctx* ctx, int which, int64_t n, const double* x, double* out);

}  // namespace fmwr
