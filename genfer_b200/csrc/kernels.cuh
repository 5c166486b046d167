// Launcher declarations for the device kernels of libgenfer_taylor (sm_100a).
#pragma once
#include <algorithm>
#include <mutex>
#include <tuple>

#include "common.hpp"

namespace gtp {

constexpr int MAXD = GTP_MAX_NDIM;

#define GTP_LAUNCH(ctx, kernel, grid, block, smem, ...)                         \
  do {                                                                          \
    const double _t0 = (ctx).hist ? ::gtp::Ctx::now() : 0.0;                    \
    kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);             \
    (ctx).launches++;                                                           \
    if ((ctx).hist) {                                                           \
      (*(ctx).hist)[#kernel]++;                                                 \
      (ctx).t_launch += ::gtp::Ctx::now() - _t0;                                \
    }                                                                           \
    GTP_CUDA(cudaGetLastError());                                               \
  } while (0)

// Lets `fn` launch with `bytes` of dynamic shared memory on `device` (the current device): raises the kernel's limit when
// it is below `bytes` and never lowers it.  The record is per (kernel, device) and shared by all contexts, which may live
// on different threads.
inline void allow_dyn_smem(const void* fn, int device, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> limit;
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = limit[{fn, device}];
  if (cur >= bytes) return;
  GTP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  cur = bytes;
}
template <class F> void allow_dyn_smem(F* fn, int device, size_t bytes) { allow_dyn_smem((const void*)fn, device, bytes); }

// Cooperative launches (persistent kernels with a grid barrier: every CTA must be resident).  Resident CTAs per SM of `fn`
// with `block` threads and `smem` bytes of dynamic shared memory on `device` (the current device), after allow_dyn_smem;
// 0 when the device has no cooperative launch or the kernel cannot be resident.  The record is per (kernel, device, block,
// smem) and shared by all contexts, which may live on different threads.
inline int coop_ctas_per_sm(const void* fn, int device, int block, size_t smem) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, int, int, size_t>, int> known;
  std::lock_guard<std::mutex> lock(mu);
  const auto key = std::make_tuple(fn, device, block, smem);
  auto it = known.find(key);
  if (it != known.end()) return it->second;
  int coop = 0, per_sm = 0;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
  if (coop) {
    allow_dyn_smem(fn, device, smem);
    GTP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, block, smem));
  }
  return known[key] = std::max(per_sm, 0);
}
// Launches `fn` cooperatively on the context's stream with one parameter struct, counted and timed as GTP_LAUNCH does
// (`tag`: its name in the GTP_LAUNCH_HIST census).
inline void coop_launch(Ctx& ctx, const void* fn, unsigned grid, int block, size_t smem, void* params, const char* tag) {
  void* args[] = {params};
  const double t0 = ctx.hist ? Ctx::now() : 0.0;
  GTP_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(block), args, smem, ctx.stream));
  ctx.launches++;
  if (ctx.hist) {
    (*ctx.hist)[tag]++;
    ctx.t_launch += Ctx::now() - t0;
  }
}

// 16-byte global -> shared copy that bypasses L1 (the DFMA product kernels stage their slabs with it)
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Generic N-D element-wise / gather kernel.  Iterates the box `ext` (after host-side coalescing of
// axes); operand A is read at a_lo+idx (valid where idx < a_ext), operand B at idx (valid where
// idx < b_ext), output written at o_lo+idx.
// ---------------------------------------------------------------------------------------------
enum EwOp : int {
  EW_COPY = 0,         // out = a * fac[idx[fax]]            (fac == nullptr -> plain copy)
  EW_ADD = 1,          // out = (0 + a?) + b?                (Add general path  :873-880)
  EW_SUB = 2,          // out = (0 + a?) - b?                (Sub general path  :928-934)
  EW_MASK = 3,         // out = keep[idx[fax]] ? a : +0.0    (taylor_polynomial_terms :394-402)
  EW_SCALE_DEV = 4,    // out = (*s) * a                     (Mul by constant   :1040-1047)
  EW_DIV_DEV = 5,      // out = a / (*s)                     (Div by constant   :1210-1213)
  EW_NEG = 6,          // out = -a                           (Neg               :902-909)
  EW_ADD_FIRST = 7,    // out = idx==0 ? a + *s : a          (Add scalar path   :862-869)
  EW_SUB_FIRST = 8,    // out = idx==0 ? a - *s : a          (Sub scalar path   :919-922)
  EW_RSUB_FIRST = 9,   // out = -(idx==0 ? a - *s : a)       (Sub scalar self   :923-926)
};

// extract_linear scan (:275-294) over a dense tensor
struct ClsParams {
  int ndim;
  unsigned shape[MAXD];
  long long str[MAXD];
  u64 total;
  unsigned all_mask;
};
// One CTA classifies the dense tensor `in` it has just written (call after the last store; contains the barriers)
// and publishes the result in `slot`, sequence number last.
__device__ __forceinline__ void cls_epilogue(const double* in, const ClsParams& p, ClsSlot* slot, unsigned long long seq) {
  __shared__ unsigned cls_sh_mask;
  __syncthreads();                 // the CTA's own stores are visible to all its threads after the barrier
  if (threadIdx.x == 0) cls_sh_mask = 0;
  __syncthreads();
  unsigned mask = 0;
  for (unsigned lin = threadIdx.x; lin < (unsigned)p.total; lin += blockDim.x) {
    const double x = in[lin];
    if (x != 0.0) {
      unsigned rem = lin;
      int nz_axis = -1, nz_count = 0;
      unsigned nz_val = 0;
      for (int d = p.ndim - 1; d >= 0; --d) {
        const unsigned q = rem / p.shape[d], i = rem - q * p.shape[d];
        rem = q;
        if (i != 0) {
          nz_count++;
          nz_axis = d;
          nz_val = i;
        }
      }
      if (nz_count >= 2) mask |= p.all_mask;
      else if (nz_count == 1) mask |= (nz_val >= 2) ? p.all_mask : (p.all_mask & ~(1u << nz_axis));
    }
  }
  if (mask) atomicOr(&cls_sh_mask, mask);
  __syncthreads();
  // ONE thread talks to host memory: payload, one system-scope fence, then the sequence number (with every thread
  // fencing and ndim threads storing slopes the epilogue cost 5.7 us per launch)
  if (threadIdx.x == 0) {
    const unsigned viol = cls_sh_mask;
    int v = -1;
    for (int d = 0; d < p.ndim; d++)
      if (p.shape[d] >= 2 && !(viol & (1u << d))) { v = d; break; }
    // No fence: each 16-byte half of the slot travels as one store (one PCIe write) together with its copy of the
    // sequence number, and the host waits for both copies -- a system-scope fence between payload and flag cost 3.8 us.
    const double first = in[0], m = v >= 0 ? in[p.str[v]] : 0.0;
    const unsigned long long tag_b = ((unsigned long long)(unsigned)seq << 32) | (unsigned)(v + 1);   // {axis_p1, seq_b}
    asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(&slot->first), "l"(__double_as_longlong(first)), "l"(seq) : "memory");
    asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(&slot->m), "l"(__double_as_longlong(m)), "l"(tag_b) : "memory");
  }
}
struct FusedClsArgs {   // kernel-side half of a fused classification (slot == nullptr: none)
  ClsSlot* slot;
  unsigned long long seq;
  ClsParams p;
};
// Host: should the single-CTA launch that writes the whole dense tensor `out` (shape) classify it?  Fills `f` and
// registers the pending result under `out`; classify() (api.cu) picks it up.
bool fused_cls_begin(Ctx& ctx, const double* out, const Shape& shape, FusedClsArgs* f);

struct EwParams {
  int ndim;
  int fax;            // axis the factor / keep arrays are indexed by (box coordinates)
  u64 total;          // prod(ext)
  unsigned ext[MAXD];
  unsigned a_ext[MAXD], b_ext[MAXD];
  long long a_str[MAXD], b_str[MAXD], o_str[MAXD];
  long long a_base, b_base, o_base;  // element offsets of (lo) corners
  const double* a;
  const double* b;
  double* out;
  const double* fac;            // device array (EW_COPY) or nullptr
  const unsigned char* keep;    // device array (EW_MASK)
  const double* s;              // device scalar, or nullptr: the scalar is s_val
  double s_val;
  FusedClsArgs cls;             // epilogue classification of the (whole, dense) output by a single-CTA launch
};

// High-level description of one operand for the host-side coalescer.
struct EwOperand {
  const double* p = nullptr;
  Shape shape;  // stored shape of the tensor (for strides)
  Shape lo;     // corner inside the tensor where box coordinate 0 maps to
  Shape valid;  // box coordinates >= valid[a] read as "absent"; empty => whole box valid
};
void launch_ew(Ctx& ctx, EwOp op, const Shape& box, const EwOperand& a, const EwOperand* b,
               double* out, const Shape& out_shape, const Shape& out_lo, int fax = -1,
               const double* fac = nullptr, const unsigned char* keep = nullptr, const double* s = nullptr,
               const double* host_tab = nullptr, int host_tab_len = 0,   // host_tab: factor table by kernel parameter
               const double* s_host = nullptr);                           // scalar by value (instead of `s`)
// derivative / binomial factor tables of at most 1024 entries built on the host (kinds 0 and 1 of launch_factors)
bool host_factors(int kind, u64 n, u64 len, double* fac, double m = 0.0);   // kind 2: powers of m

void launch_fill(Ctx& ctx, double* dst, u64 n, double value);
// fused mul_linear / mul_var (:589-623) on the (outer, xlen, inner) view of the variable's axis; out has olen (xlen or xlen + 1) slices
void launch_mul_linear(Ctx& ctx, const double* x, double* out, u64 outer, u64 xlen, u64 olen, u64 inner, double c, double m,
                       const Shape& out_shape);
// fac[k], k < len:  kind 0: falling factorials (n+k)!/k!  (derivative :472-479)
//                   kind 1: binomials C(n+k,k)            (taylor_expansion_of_coeff :499-507)
//                   kind 2: powers (*m)^k                 (subst_var linear path :557-565)
void launch_factors(Ctx& ctx, int kind, u64 n, u64 len, const double* m, double* fac);

// shift_down (:514-536) on the (outer, len, inner) view of axis v.  out has (outer, out_len, inner).
// `last_axis`: v is the last stored axis (ndarray sums those lanes with its 8-way unrolled fold).
void launch_shift_down(Ctx& ctx, const double* in, double* out, u64 outer, u64 len, u64 inner, u64 n,
                       bool last_axis);
// evaluate_all_one (:583-586): *out_dev = sum of all n elements
void launch_sum_all(Ctx& ctx, const double* in, u64 n, double* out_dev);
// classification for extract_linear (:275-294): writes Readback{viol_mask, vals[0]=first} to rb_dev
void launch_classify(Ctx& ctx, const double* in, const Shape& shape, Readback* rb_dev);
// Small tensors (<= 8192 coefficients): ONE single-CTA kernel that writes the classification straight into the mapped
// pinned page and bumps its sequence number; the host spins on it (no memset, no D2H copy, no stream synchronise).
// Returns false if the tensor is too large for this path.
bool classify_small_zero_copy(Ctx& ctx, const double* in, const Shape& shape);
// rb_dev->flag = 1 iff every element compares == (IEEE)
void launch_eq(Ctx& ctx, const double* a, const double* b, u64 n, Readback* rb_dev);
// out[i] = i < len ? in[i*stride] : 0   for i < count
void launch_gather_strided(Ctx& ctx, const double* in, u64 stride, u64 len, u64 count, double* out);

// ---------------------------------------------------------------------------------------------
// Product (kernels_mul.cu).  Computes output rows k0 = row_begin + i*row_step (i < row_count) of
// X (*) Y truncated to rshape; row i lands at out + i*prod(rshape[1:]).  If `accumulate` the rows
// are added to (sign > 0) / subtracted from what is there; otherwise overwritten.
// ---------------------------------------------------------------------------------------------
struct MulArgs {
  int ndim;
  Shape xs, ys, rs;
  const double* x = nullptr;
  const double* y = nullptr;
  double* out = nullptr;
  u64 row_begin = 0, row_step = 1, row_count = 0;
  std::vector<u64> rows;  // explicit leading-axis row list (overrides begin/step/count when non-empty)
  bool accumulate = false;
  double sign = 1.0;
};
void launch_mul(Ctx& ctx, const MulArgs& a);
// The product kernel launch_mul runs for `a` (its plan, nothing launched): 0 the reference-order family (reference-order
// kernel, small-operand products, axis convolution: all bit-exact), 2 / 3 the blocked / sliding DFMA kernel, 6 / 7 the same
// after zero-extending odd extents.
int mul_kernel_kind(const Ctx& ctx, const MulArgs& a);
double mul_macs(const Shape& xs, const Shape& ys, const Shape& rs);
double args_macs(const MulArgs& a);   // MACs of the rows this launch computes
// Products below this many MACs stay on the reference-order kernel (bit-exact, and launch-bound anyway); above it the
// DFMA kernels run even when only a few slabs exist (their units split the j box, so a handful of slabs still fills the SMs)
constexpr double DFMA_MIN_MACS = 1 << 20;

// Host plan path of the DFMA product kernels (the 2x2-blocked k_mul_blk and the sliding k_mul_slide / k_mul_slide16).
// Chunk length of a last axis of `l` doubles: the longest of 16, 14, 12, 10, 8 that divides it; 0: none does.
u64 dfma_chunk(u64 l);
// `doubles` rounded up to an even count whose half is odd: shared-memory strides of an odd number of 16-byte groups put
// the planes / staged slabs that lockstep lanes read into different bank groups.
inline u64 odd_groups(u64 doubles) {
  doubles = (doubles + 1) / 2 * 2;
  if ((doubles / 2) % 2 == 0) doubles += 2;
  return doubles;
}
// Work units {packed output slab index, q0, q1, k along A axis 0}: each output slab of the A axes (extents axs / ays / ars
// of X, Y and Z; axis 0 walks the launch's rows) splits its box of (X slab, Y slab) pairs into chunks [q0, q1) of whole
// rounds of G pairs.  Units run at least 8 rounds unless that leaves some of the `slots` resident CTAs idle.  Sorted
// longest first (LPT).
std::vector<uint4> dfma_units(const MulArgs& a, const Shape& axs, const Shape& ays, const Shape& ars, int G, u64 slots);
// Device arrays of a cached plan; the kernel-specific plans derive from it.
struct DfmaPlan {
  BufP table, units;   // step table (uint2 entries) and work units (uint4)
  unsigned n_units = 0;
};
// The entry of `cache` (a context's plan slot) for this product's shapes and rows and the caller's `extra` word.  Empty on
// a miss: the caller builds the plan and stores it there.  A cache that holds more than 64 plans is cleared first.
std::shared_ptr<void>& dfma_plan_slot(std::shared_ptr<void>& cache, const MulArgs& a, u64 extra);
// Copies the step table and the units to new device arrays of `pl` (empty arrays are not copied) and waits for the copy.
void dfma_upload(Ctx& ctx, DfmaPlan* pl, const std::vector<uint2>& table, const std::vector<uint4>& units);

// The terms of a small operand (at most 32 coefficients, extents <= 255) in a product or a Horner step: coefficient sidx[t]
// pairs with the big operand at k - m[t] (m over the `ne` effective axes `eff`; the small operand has extent 1 on every
// other axis).  Sorted in the reference's visiting order, ascending X index: ascending m when the small operand is X,
// descending m (`descending`) when it is Y; group_start[t] marks the first term of each group of equal outer offsets.
constexpr int SMALL_MAXT = 32, SMALL_MAXE = 8;
struct SmallTerms {
  int nt;
  unsigned char m[SMALL_MAXT][SMALL_MAXE];   // zero beyond the effective axes
  unsigned short sidx[SMALL_MAXT];
  unsigned char group_start[SMALL_MAXT];
};
SmallTerms small_terms(const Shape& ss, const int* eff, int ne, bool descending);

void fp64_peak_probe(Ctx& ctx, int kind, int iters, double* flops, double* ms);

// ---------------------------------------------------------------------------------------------
// Recurrences (kernels_rec.cu)
// ---------------------------------------------------------------------------------------------
// Division by a divisor that is non-constant along exactly one axis: (outer, len, inner) views.
// x has x_len slices along the axis (zero beyond), y has y_len coefficients, r has r_len slices.
// Per lane exactly the reference's operation order (:1170-1191 specialised), bit-exact.
void launch_div_axis(Ctx& ctx, const double* x, const double* y, double* r, u64 outer, u64 inner,
                     u64 x_len, u64 y_len, u64 r_len, const Shape& xshape_full, const Shape& rshape_full, int axis);
// General N-D division by total-degree wavefronts.
void launch_div_general(Ctx& ctx, const double* x, const Shape& xs, const double* y, const Shape& ys,
                        double* r, const Shape& rs);
// Device-resident N-D recurrences (kernels_wave.cu): general division (op 0, y = divisor), exp (1), log (2) as ONE
// cooperative kernel walking the leaf levels.  `exact`: exp only -- reference summation order, bit-identical.
// Returns false when the shapes are outside its domain (fewer than two non-unit result axes, ...).
bool launch_rec_wave(Ctx& ctx, int op, const double* x, const Shape& xs, const double* y, const Shape& ys, double* r,
                     const Shape& rs, bool exact, const double* seed = nullptr);
// Fused Horner loop of subst_var (kernels_horner.cu): steps i_top .. 0 of `res = res * subst + self.slice(v, i)` in ONE
// cooperative kernel, for a substitution of 2..32 coefficients.  Bit-identical to the per-operator steps.  false: outside
// its domain (the caller continues step by step).
bool launch_horner(Ctx& ctx, const double* self, const Shape& self_shape, u64 v, const Shape& d, const double* subst,
                   const Shape& sshape, const double* res, const Shape& rshape, u64 i_top, BufP* out_buf, Shape* out_shape);
// 1-D exp / log recurrences (exp_1d :1271-1283, log_1d :1319-1333) on contiguous vectors
// `seed` (host pointer or nullptr): exp / log of the constant term x[0] evaluated by the host's libm, used when the host
// already knows x[0] -- the reference calls the same libm (number/f64.rs:53-62), so the result is then bit-identical;
// nullptr: CUDA's exp / log (<= 1 ulp) on the device, no synchronisation.
void launch_exp_1d(Ctx& ctx, const double* x, u64 xlen, double* r, u64 n, const double* seed = nullptr);
void launch_log_1d(Ctx& ctx, const double* x, u64 xlen, double* r, u64 n, const double* seed = nullptr);
// r[0] = exp(x[0]) / log(x[0])  (scalar leaf :1289-1291, :1339-1341)
void launch_scalar_fn(Ctx& ctx, int fn, const double* x, double* r, const double* seed = nullptr);
// out[i] = in[i] * k   or   in[i] / k   (k an integer-valued double; :1309, :1315, :1364, :1374, :1384)
void launch_scale_const(Ctx& ctx, const double* in, double* out, u64 n, double k, bool divide);
// rows j = 0..rows-1 of `in` (row length `inner`) scaled by (j + j0):  out[j,:] = in[j,:] * (j+j0)
void launch_scale_rows(Ctx& ctx, const double* in, double* out, u64 rows, u64 inner, u64 j0, bool left);

// ---------------------------------------------------------------------------------------------
// Univariate TaylorExpansion kernels (univariate.cu)
// ---------------------------------------------------------------------------------------------
void uni_mul(Ctx& ctx, const double* u, const double* w, double* r, u64 order);          // :376-386
void uni_div(Ctx& ctx, const double* u, bool u_const, const double* w, double* r, u64 order);  // :409-436
void uni_exp(Ctx& ctx, const double* c, double* r, u64 order);                            // :153-164
void uni_log(Ctx& ctx, const double* c, double* r, u64 order);                            // :172-185
// r[i] = op(a[i or 0], b[i or 0]) element-wise family for the Constant/Polynomial combinations (op: UniEw)
void uni_ew(Ctx& ctx, int op, const double* a, bool a_bcast, const double* b, bool b_bcast, double* r, u64 n);
void uni_teoc(Ctx& ctx, const double* in, double* out, u64 n, u64 len);                   // :78-87
void uni_factorial_times(Ctx& ctx, const double* in, u64 order, double* out);             // :47-51

// uni_ew's operations
enum UniEw : int {
  UEW_ADD = 0, UEW_SUB = 1, UEW_MUL = 2, UEW_DIV = 3, UEW_NEG = 4,
  UEW_ADD_FIRST = 5,    // r = a; r[0] += b
  UEW_SUB_FIRST = 6,    // r = a; r[0] -= b
  UEW_RSUB_FIRST = 7,   // r = -a; r[0] += b
  UEW_MAX = 8,          // a > b ? a : b (Constants only)
};
// The kernel that runs one univariate op
enum UniKind : int { UK_EW = 0, UK_MUL, UK_DIV, UK_EXP, UK_LOG, UK_SCALAR_EXP, UK_SCALAR_LOG };
// What an op (GTU_ADD ... GTU_MAX) does to operands of the given variants and lengths (n: 1 for a Constant): the result's
// variant and length and the kernel that computes it.  The kernel's operands are (a, b), or (b, a) when `swap`; a_b / b_b
// broadcast element 0 of the kernel's first / second operand (UK_DIV: a_b = the dividend is a Constant).  Throws the
// reference's errors: GTP_ERR_INDEX for Max of a Polynomial, GTP_ERR_ARG for a quotient above order 2048.
struct UniPlan {
  bool is_const = true;
  u64 n = 1;
  int kind = UK_EW;
  int ew = 0;
  bool swap = false, a_b = false, b_b = false;
};
UniPlan uni_plan(int op, bool a_const, u64 a_n, bool b_const, u64 b_n);
// runs a plan with the per-op kernels; b may be null for unary ops
void uni_run(Ctx& ctx, const UniPlan& p, const double* a, const double* b, double* r);

// One instruction of a univariate program (k_uni_program): a plan with its kernel operands resolved to arena offsets
constexpr unsigned UNI_NONE = 0xffffffffu;
struct UniIns {
  unsigned a, b, r;   // arena offsets (doubles) of the kernel's first and second operand (UNI_NONE: none) and of the result
  unsigned n;         // result length
  unsigned char kind, ew, a_b, b_b;
  unsigned pad;
};
static_assert(sizeof(UniIns) == 24, "UniIns is packed into a double-aligned upload");
// ins / lvl / outs / arena are device pointers; lvl has nlevels * nwarps + 1 entries, outs n_out (src, len, dst) triples
void uni_program_launch(Ctx& ctx, const UniIns* ins, const unsigned* lvl, int nlevels, int nwarps, const unsigned* outs, int n_out,
                        double* arena);

}  // namespace gtp
