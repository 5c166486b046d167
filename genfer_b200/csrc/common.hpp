// Internal types of libgenfer_taylor: context, immutable ref-counted device buffers, handles.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <map>
#include <unordered_map>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/genfer_taylor.h"

namespace gtp {

using u64 = uint64_t;
constexpr u64 UNB = GTP_UNBOUNDED;
using Shape = std::vector<u64>;

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
#define GTP_CHECK(cond, code, msg)                    \
  do {                                                \
    if (!(cond)) throw ::gtp::Error((code), (msg));   \
  } while (0)
#define GTP_CUDA(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      throw ::gtp::Error(_e == cudaErrorMemoryAllocation ? GTP_ERR_OOM : GTP_ERR_CUDA,              \
                         std::string(#expr) + ": " + cudaGetErrorString(_e));                       \
  } while (0)

inline u64 prod(const Shape& s) {
  u64 p = 1;
  for (u64 x : s) p *= x;
  return p;
}
inline u64 sat_sub(u64 a, u64 b) { return a > b ? a - b : 0; }

struct Ctx;

// The stream outlives the context for as long as any buffer allocated on it is alive.
struct StreamCore {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own = false;
  cudaMemPool_t pool = nullptr;   // private stream-ordered pool of this context (nullptr: the device's default pool)
  // Size-class cache in front of the stream-ordered pool: every buffer lives on this one stream, so a released block can
  // be handed out again at once.  Requests are rounded up to classes of 1/8 octave, which lets the ever-growing tensors of
  // a Horner / recurrence loop reuse each other's blocks (each new size used to make the pool map fresh physical memory:
  // cudaMallocAsync was 0.46 s of a 0.55 s run of the population models) and replaces a ~0.7 us driver call per
  // operation by a vector pop.
  std::unordered_map<u64, std::vector<void*>> free_cache;
  u64 cached_bytes = 0;
  static constexpr u64 CACHE_CAP = 96ull << 30;
  static u64 size_class(u64 bytes) {
    if (bytes <= 4096) return (bytes + 255) / 256 * 256;
    u64 p = 1;
    while ((p << 1) <= bytes) p <<= 1;          // largest power of two <= bytes
    const u64 step = p >> 3;
    return (bytes + step - 1) / step * step;
  }
  void release(void* d, u64 cls_bytes) {
    if (cls_bytes && cached_bytes + cls_bytes <= CACHE_CAP) {
      free_cache[cls_bytes].push_back(d);
      cached_bytes += cls_bytes;
    } else {
      cudaFreeAsync(d, stream);
    }
  }
  void* take(u64 cls_bytes) {
    auto it = free_cache.find(cls_bytes);
    if (it == free_cache.end() || it->second.empty()) return nullptr;
    void* d = it->second.back();
    it->second.pop_back();
    cached_bytes -= cls_bytes;
    return d;
  }
  void trim() {   // give everything back to the pool (out of memory, context teardown)
    for (auto& kv : free_cache)
      for (void* d : kv.second) cudaFreeAsync(d, stream);
    free_cache.clear();
    cached_bytes = 0;
  }
  ~StreamCore() {
    if (stream) {
      trim();
      cudaStreamSynchronize(stream);
    }
    if (pool) cudaMemPoolDestroy(pool);
    if (own && stream) cudaStreamDestroy(stream);
  }
};

// Slots of two doubles in mapped pinned host memory for scalars and `x + eps_v` variables (the tensors of one or two
// coefficients every program creates by the hundred thousand: constants, probabilities, variables).  The host writes the
// value directly -- no kernel launch, no copy -- and kernels read it over PCIe through the same (unified) address.  A
// released slot may still be read by kernels in flight, so it is recycled only after a stream synchronise, which happens
// once per ~10^6 releases.
struct ScalarPool {
  static constexpr size_t SLOTS_PER_BLOCK = 1 << 16, MAX_BLOCKS = 16;
  std::shared_ptr<StreamCore> core;
  std::vector<double*> blocks, free_slots, pending;
  bool disabled = false;
  double* acquire() {
    if (disabled) return nullptr;
    if (free_slots.empty()) {
      if (blocks.size() < MAX_BLOCKS || pending.empty()) {
        double* b = nullptr;
        if (cudaHostAlloc((void**)&b, SLOTS_PER_BLOCK * 16, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
          cudaGetLastError();
          disabled = blocks.empty();
          if (disabled || pending.empty()) return nullptr;
        } else {
          void* dp = nullptr;
          if (cudaHostGetDevicePointer(&dp, b, 0) != cudaSuccess || dp != (void*)b) {   // no unified addressing
            cudaGetLastError();
            cudaFreeHost(b);
            disabled = true;
            return nullptr;
          }
          blocks.push_back(b);
          for (size_t i = SLOTS_PER_BLOCK; i-- > 0;) free_slots.push_back(b + 2 * i);
        }
      }
      if (free_slots.empty()) {
        if (cudaStreamSynchronize(core->stream) != cudaSuccess) return nullptr;
        free_slots.swap(pending);
      }
    }
    double* p = free_slots.back();
    free_slots.pop_back();
    return p;
  }
  void release(double* p) { pending.push_back(p); }
  ~ScalarPool() {
    if (core && core->stream) cudaStreamSynchronize(core->stream);
    for (double* b : blocks) cudaFreeHost(b);
  }
};

// Immutable device buffer.  Freed stream-ordered (cudaFreeAsync) when the last handle drops it.
struct Buf {
  double* d = nullptr;
  u64 n = 0;       // doubles
  bool owned = true;
  std::shared_ptr<StreamCore> core;
  std::shared_ptr<ScalarPool> pool;   // set: `d` is a slot of the scalar pool (host-visible)
  u64 cls_bytes = 0;                  // size class the block was allocated with (0: not from the cache)
  ~Buf() {
    if (pool) pool->release(d);
    else if (owned && d && core) core->release(d, cls_bytes);
  }
};
using BufP = std::shared_ptr<Buf>;

// Pinned read-back page layout (host-visible, written by kernels / D2H copies)
struct Readback {
  unsigned int viol_mask;  // classify: bit v set <=> axis v is NOT a linear axis
  unsigned int flag;       // generic boolean result (eq / any)
  double vals[64];         // c, m, sums, gathered scalars ...
  volatile unsigned long long seq;  // written LAST by the single-CTA classify kernel (zero-copy path): host spins on it
};

// Classification written by the PRODUCING kernel (single-CTA element-wise kernels run the extract_linear scan over
// their own output as an epilogue): one slot of a ring in mapped pinned memory per fused launch.  `seq` is written last.
struct ClsSlot {                   // two 16-byte halves, each written by ONE vector store that carries the sequence number
  double first;                    // coeffs.first()
  volatile unsigned long long seq_a;
  double m;                        // coefficient at e_v of the linear axis
  unsigned axis_p1;                // 0: not linear, else 1 + the linear axis v
  volatile unsigned seq_b;         // low 32 bits of the sequence number
};
struct FusedCls {
  unsigned long long seq = 0;
  Shape shape;
};

// ---- multi-GPU group (SURVEY 8e): one context = one stream + one NCCL communicator --------------------------------
// NCCL is loaded with dlopen when a group context is created (group.cu): the library has no link-time dependency on it
// and single-GPU use never touches it.
struct NcclApi;
struct Group {
  int rank = 0, world = 1;
  void* comm = nullptr;                 // ncclComm_t
  std::shared_ptr<NcclApi> api;
  u64 threshold = 10000000;             // products with at least this many output coefficients are partitioned (north_star)
  u64 partitioned_products = 0, gathers = 0;   // statistics (bench / tests)
  ~Group();
};

struct Ctx {
  int device = 0;
  std::shared_ptr<Group> group;        // null: single-GPU context
  std::shared_ptr<StreamCore> core;
  cudaStream_t stream = nullptr;  // == core->stream
  int sm_count = 148;
  std::string err;
  Readback* rb_host = nullptr;  // pinned
  Readback* rb_dev = nullptr;   // device scratch mirrored into rb_host by cudaMemcpyAsync
  unsigned int* counter_dev = nullptr;  // "last block" tickets etc.
  double* gather_host = nullptr;        // pinned, for gtp_gather_axis / to_host staging
  u64 gather_cap = 0;
  u64 launches = 0;
  std::map<std::string, u64>* hist = nullptr;   // per-kernel launch counts (GTP_LAUNCH_HIST=1; printed when the context is destroyed)
  u64 rb_seq = 0;               // sequence number of the last zero-copy read-back request
  Readback* rb_host_dev = nullptr;  // device alias of rb_host (mapped pinned memory)
  int fast_mul = 1;  // 0: reference-order kernel only, 1: auto, 2: force the blocked kernel even on tiny products (tests)
  std::shared_ptr<void> blk_plans;   // per-context caches of DFMA product plans (kernels_mul_blk.cu, dfma_plan_slot)
  std::shared_ptr<void> slide_plans; // same for kernels_mul_slide.cu
  std::shared_ptr<void> wave_tables; // level tables of the device-resident recurrences (kernels_wave.cu)
  bool bulk_products = false;        // also run plain small-operand products on the row-staged kernel (A/B; slower than the gather kernel)
  bool use_direct = true;            // row-walking plain-load variant of the Horner step (k_horner_direct), tried before the bulk-copy one
  bool direct_products = true;       // plain small-operand products with rows of at least 192 coefficients on k_horner_direct (0.119 against 0.137 ms)
  bool direct_products_all = false;  // ... with any row length (A/B: the four-coefficient gather kernel is faster on short rows)
  u64 direct_min = 1u << 17;         // smallest final tensor (coefficients) that goes to k_horner_direct (GTP_DIRECT_MIN)
  int direct_ctas = 4;               // resident CTAs per SM for HBM-sized k_horner_direct launches (GTP_DIRECT_CTAS)
  bool use_bulk = true;              // row-staged (bulk-copy / TMA) variant of the Horner step and the small-operand product (A/B tests)
  bool use_pad = true;               // zero-extend odd-shaped dense products to the DFMA kernels' extents (A/B tests)
  bool use_axis = true;              // 1-d operand x N-d tensor: batched axis convolution kernel (false: reference-order kernel; A/B tests)
  bool use_horner = true;            // fused Horner loop of subst_var for substitutions of <= 32 coefficients (A/B tests)
  bool use_wave = true;              // device-resident N-D div / exp / log (false: host loops of product launches; A/B tests)
  bool use_slide = true;             // sliding 1x2 kernel for dense cube slabs (false: 2x2-blocked kernel everywhere)
  int slide_tile = 0;                // 0: auto; 4 / 8: force the plane-tiled sliding plan with that many planes per slab
  bool slide_runs = true;            // whole 16^3 slabs on the run-granular sliding kernel (false: the step-table one; A/B)
  bool stencil_v4 = true;            // stencil kernel: four coefficients per thread (false: one; A/B tests, bit 512)
  bool use_stencil = true;           // small-operand stencil product kernel (false: reference-order kernel; A/B tests)
  bool fuse_mul_linear = true;       // one-pass mul_linear kernel (false: the reference's composition, for A/B tests)

  std::shared_ptr<ScalarPool> scalars;   // created with the context
  static constexpr unsigned CLS_RING = 1 << 16;
  ClsSlot* cls_ring = nullptr;           // mapped pinned (host pointer == device pointer), CLS_RING slots
  unsigned long long cls_seq = 0;        // last sequence number handed to a fused launch (slot = seq % CLS_RING)
  std::unordered_map<const double*, FusedCls> fused_cls;   // result buffer -> its in-flight / finished classification
  u64 fused_hits = 0;
  double t_spin = 0, t_alloc = 0, t_launch = 0;   // seconds, only measured when `hist` is on (GTP_LAUNCH_HIST=1)
  static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
  BufP alloc(u64 n_doubles);
  BufP alloc_host_visible(const double* vals, int n);   // n <= 2: a scalar-pool slot holding vals (nullptr: pool unavailable)
  void sync() { GTP_CUDA(cudaStreamSynchronize(stream)); }
  // gather_host with room for n doubles; grows it (the old block must not be in use by a pending copy)
  double* host_staging(u64 n) {
    if (gather_cap < n) {
      if (gather_host) cudaFreeHost(gather_host);
      gather_host = nullptr;
      gather_cap = 0;
      GTP_CUDA(cudaMallocHost((void**)&gather_host, std::max<u64>(n, 1024) * sizeof(double)));
      gather_cap = std::max<u64>(n, 1024);
    }
    return gather_host;
  }
};

// Cached data-dependent classification of a handle (multivariate_taylor.rs:262-294, :643-655)
struct ClassInfo {
  bool known = false;
  bool linear = false;  // extract_linear() is Some
  double c = 0, m = 0;  // if linear
  u64 v = 0;            // if linear
  double first = 0;     // coeffs.first()
};

}  // namespace gtp

namespace gtp {
// A polynomial whose coefficients are distributed over the ranks of a group context: either the folded-cyclic leading-axis
// ROWS a partitioned product left on this rank, or this rank's contiguous BLOCK of leading-axis slices (an operand
// uploaded in shards).  `shape` of the handle is always the FULL shape.  The first consumer that needs the whole tensor
// replicates it (NCCL broadcasts / all-gather on the context's stream) and caches the result here, shared by all clones.
struct ShardState {
  enum Kind { ROWS, BLOCK } kind = ROWS;
  Ctx* ctx = nullptr;
  std::shared_ptr<Group> group;
  BufP local;                    // ROWS: rows[i] at local + i * row_elems;  BLOCK: the (zero-padded) block of `block` slices
  const double* local_ptr = nullptr;   // BLOCK built over caller-owned device memory (gtp_from_device_block)
  std::vector<u64> rows;         // ROWS: this rank's leading-axis rows, ascending
  u64 n_rows = 0, row_elems = 0, block = 0;
  BufP full;                     // set once replicated
};
const double* replicate(const ShardState& s);   // group.cu; idempotent
}  // namespace gtp

// The opaque handle types of the C ABI
struct gtp_poly {
  gtp::BufP buf;
  gtp::u64 off = 0;  // element offset of this polynomial inside buf (prefix views)
  gtp::Shape shape;    // coeffs.shape()
  gtp::Shape degrees;  // degrees_p1
  std::shared_ptr<gtp::ClassInfo> cls = std::make_shared<gtp::ClassInfo>();  // shared by O(1) clones of the same data
  std::shared_ptr<gtp::ShardState> shard;   // set: distributed over a group context (buf is null until replicated)
  const double* ptr() const { return shard ? gtp::replicate(*shard) + off : buf->d + off; }
  gtp::u64 len() const { return gtp::prod(shape); }
  int ndim() const { return (int)shape.size(); }
};

struct gtu_series {
  bool is_const = false;
  gtp::BufP buf;  // 1 element for Constant, `n` for Polynomial
  gtp::u64 n = 1;
  const double* ptr() const { return buf->d; }
};

struct gtp_ctx : gtp::Ctx {};
