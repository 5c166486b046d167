// Device kernels for the univariate TaylorExpansion<F64> (src/univariate_taylor.rs).  Series are
// short (order <= limit <= 1000, src/main.rs:30), so every op is one small launch, or one instruction
// of a recorded program (k_uni_program).  Products, quotients and the element-wise family keep the
// reference's operation order with separately rounded multiply/add and are bit-identical to it;
// exp/log use a fixed 256-way reduction for long sums.
//
// Each op's arithmetic is written once, as a __device__ function over a "team" of threads: the per-op
// kernels run it on their own geometry, k_uni_program on one warp.  The rounding sequence of every
// coefficient depends only on the op, never on the team, so both give the same bits.
#include "kernels.cuh"

namespace gtp {

constexpr int UNI_T = 256;       // the 256 partial sums of the long exp / log sums; k_uni_div's block
constexpr u64 UNI_MAX_DIV = 2048;

struct BlockTeam {   // the whole CTA of UNI_T threads
  static constexpr unsigned SIZE = UNI_T;
  __device__ unsigned rank() const { return threadIdx.x; }
  __device__ void sync() const { __syncthreads(); }
};
struct WarpTeam {    // one warp of k_uni_program
  static constexpr unsigned SIZE = 32;
  unsigned lane;
  __device__ unsigned rank() const { return lane; }
  __device__ void sync() const { __syncwarp(); }
};

// Operands of the team functions are plain pointers on purpose: in k_uni_program they point into the arena that earlier
// levels of the same launch wrote, so the read-only (non-coherent) load path must not be used for them.

// Mul :376-386 -- result[k] = fold_{j=0..k}(sum + us[j]*ws[k-j]); each k on one thread, same order.
__device__ __forceinline__ void uni_mul_team(u64 rank, u64 size, const double* u, const double* w, double* r, u64 order) {
  for (u64 k = rank; k < order; k += size) {
    double sum = 0.0;
    for (u64 j = 0; j <= k; j++) sum = __dadd_rn(sum, __dmul_rn(u[j], w[k - j]));
    r[k] = sum;
  }
}

// Element-wise family covering the Constant/Polynomial combinations of AddAssign :277-306,
// SubAssign :330-362, Mul-by-constant :370-375, Div-by-constant :403-408, Neg :308-319, and F64::max
// of two Constants (number/f64.rs:77-84).
__device__ __forceinline__ void uni_ew_team(u64 rank, u64 size, int op, const double* a, int a_b, const double* b, int b_b,
                                            double* r, u64 n) {
  for (u64 i = rank; i < n; i += size) {
    double x = a[a_b ? 0 : i];
    double y = b ? b[b_b ? 0 : i] : 0.0;
    double v;
    switch (op) {
      case UEW_ADD: v = __dadd_rn(x, y); break;
      case UEW_SUB: v = __dsub_rn(x, y); break;
      case UEW_MUL: v = __dmul_rn(x, y); break;
      case UEW_DIV: v = __ddiv_rn(x, y); break;
      case UEW_NEG: v = -x; break;
      case UEW_ADD_FIRST: v = (i == 0) ? __dadd_rn(x, y) : x; break;     // coeffs[0] += rhs
      case UEW_SUB_FIRST: v = (i == 0) ? __dsub_rn(x, y) : x; break;     // coeffs[0] -= rhs
      case UEW_RSUB_FIRST: v = (i == 0) ? __dadd_rn(-x, y) : -x; break;  // ws = -ws; ws[0] += c   (:340-344)
      default: v = x > y ? x : y; break;                                 // UEW_MAX
    }
    r[i] = v;
  }
}

// Div :409-436 -- scale = 1/ws[0]; result[k] = scale * fold_{i<k}(init_k, sum - result[i]*ws[k-i]).
// Column oriented: r[k] holds the running sum of a pending k; when r[i] is final every pending k
// subtracts r[i]*ws[k-i], so each sum sees i ascending, i.e. the reference's fold order.  Row k is
// owned by rank k % SIZE, which also finalises it.
template <class Team>
__device__ __forceinline__ void uni_div_team(const Team& t, const double* u, int u_const, const double* w, double* r, u64 order) {
  if (order == 0) return;
  const double scale = __ddiv_rn(1.0, w[0]);
  for (u64 k = t.rank(); k < order; k += Team::SIZE) r[k] = u_const ? 0.0 : u[k];
  for (u64 i = 0; i < order; i++) {
    if (i % Team::SIZE == t.rank()) r[i] = (i == 0) ? __dmul_rn(u_const ? u[0] : r[0], scale) : __dmul_rn(scale, r[i]);
    t.sync();
    const double ri = r[i];
    u64 k = i + 1 + (t.rank() + Team::SIZE - (i + 1) % Team::SIZE) % Team::SIZE;   // first owned row above i
    for (; k < order; k += Team::SIZE) r[k] = __dsub_rn(r[k], __dmul_rn(ri, w[k - i]));
  }
  t.sync();
}

// The long sums of exp / log: sum over j in [lo, hi) of term(j) as UNI_T strided fma partial sums, a shuffle tree per
// 32 partials and a fixed tree over the 8 warp sums.  A team of SIZE threads runs UNI_T / SIZE partials per thread
// (partial v on rank v % SIZE), so every team produces the same bits.  `sh` holds 8 doubles; the sum is valid on rank 0.
template <class Team, class Term>
__device__ __forceinline__ double uni_team_sum(const Team& t, u64 lo, u64 hi, Term term, double* sh) {
  constexpr unsigned VPT = UNI_T / Team::SIZE;
#pragma unroll
  for (unsigned q = 0; q < VPT; q++) {
    const unsigned v = t.rank() + Team::SIZE * q;
    double part = 0.0;
    for (u64 j = lo + v; j < hi; j += UNI_T) part = term(j, part);
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if ((v & 31) == 0) sh[v >> 5] = part;
  }
  t.sync();
  double s = 0.0;
  if (t.rank() == 0) s = ((sh[0] + sh[4]) + (sh[2] + sh[6])) + ((sh[1] + sh[5]) + (sh[3] + sh[7]));
  return s;
}

// exp :153-164 -- res[k] = (sum_{j=1..k} res[k-j]*coeffs[j]*j) / k
template <class Team>
__device__ __forceinline__ void uni_exp_team(const Team& t, const double* c, double* r, u64 order, double* sh) {
  if (order == 0) return;
  if (t.rank() == 0) r[0] = exp(c[0]);
  t.sync();
  for (u64 k = 1; k < order; k++) {
    double sum = 0.0;
    if (k <= 32) {
      if (t.rank() == 0)
        for (u64 j = 1; j <= k; j++) sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(r[k - j], c[j]), (double)(unsigned)j));
    } else {
      sum = uni_team_sum(t, 1, k + 1, [&](u64 j, double p) { return fma(__dmul_rn(r[k - j], c[j]), (double)(unsigned)j, p); }, sh);
    }
    if (t.rank() == 0) r[k] = __ddiv_rn(sum, (double)(unsigned)k);
    t.sync();
  }
}

// log :172-185 -- res[k] = (coeffs[k]*k - sum_{j=1..k-1} coeffs[k-j]*res[j]*j) / coeffs[0] / k
template <class Team>
__device__ __forceinline__ void uni_log_team(const Team& t, const double* c, double* r, u64 order, double* sh) {
  if (order == 0) return;
  if (t.rank() == 0) r[0] = log(c[0]);
  t.sync();
  const double c0 = c[0];
  for (u64 k = 1; k < order; k++) {
    double sum = 0.0;
    if (k <= 33) {
      if (t.rank() == 0)
        for (u64 j = 1; j < k; j++) sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(c[k - j], r[j]), (double)(unsigned)j));
    } else {
      sum = uni_team_sum(t, 1, k, [&](u64 j, double p) { return fma(__dmul_rn(c[k - j], r[j]), (double)(unsigned)j, p); }, sh);
    }
    if (t.rank() == 0) {
      double kk = (double)(unsigned)k;
      r[k] = __ddiv_rn(__ddiv_rn(__dsub_rn(__dmul_rn(c[k], kk), sum), c0), kk);
    }
    t.sync();
  }
}

// ---- per-op kernels ----------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(128) k_uni_mul(const double* __restrict__ u, const double* __restrict__ w, double* r, u64 order) {
  uni_mul_team((u64)blockIdx.x * blockDim.x + threadIdx.x, (u64)gridDim.x * blockDim.x, u, w, r, order);
}
void uni_mul(Ctx& ctx, const double* u, const double* w, double* r, u64 order) {
  if (order == 0) return;
  GTP_LAUNCH(ctx, k_uni_mul, (unsigned)((order + 127) / 128), 128, 0, u, w, r, order);
}

__global__ void __launch_bounds__(UNI_T) k_uni_div(const double* __restrict__ u, int u_const, const double* __restrict__ w,
                                                  double* r, u64 order) {
  uni_div_team(BlockTeam{}, u, u_const, w, r, order);
}
void uni_div(Ctx& ctx, const double* u, bool u_const, const double* w, double* r, u64 order) {
  GTP_CHECK(order <= UNI_MAX_DIV, GTP_ERR_ARG, "univariate order > 2048 not supported");
  if (order == 0) return;
  GTP_LAUNCH(ctx, k_uni_div, 1, UNI_T, 0, u, u_const ? 1 : 0, w, r, order);
}

__global__ void __launch_bounds__(UNI_T) k_uni_exp(const double* __restrict__ c, double* r, u64 order) {
  __shared__ double sh[UNI_T / 32];
  uni_exp_team(BlockTeam{}, c, r, order, sh);
}
__global__ void __launch_bounds__(UNI_T) k_uni_log(const double* __restrict__ c, double* r, u64 order) {
  __shared__ double sh[UNI_T / 32];
  uni_log_team(BlockTeam{}, c, r, order, sh);
}
void uni_exp(Ctx& ctx, const double* c, double* r, u64 order) {
  if (order) GTP_LAUNCH(ctx, k_uni_exp, 1, UNI_T, 0, c, r, order);
}
void uni_log(Ctx& ctx, const double* c, double* r, u64 order) {
  if (order) GTP_LAUNCH(ctx, k_uni_log, 1, UNI_T, 0, c, r, order);
}

__global__ void __launch_bounds__(256) k_uni_ew(int op, const double* __restrict__ a, int a_b, const double* __restrict__ b, int b_b,
                                               double* r, u64 n) {
  uni_ew_team((u64)blockIdx.x * blockDim.x + threadIdx.x, (u64)gridDim.x * blockDim.x, op, a, a_b, b, b_b, r, n);
}
void uni_ew(Ctx& ctx, int op, const double* a, bool a_bcast, const double* b, bool b_bcast, double* r, u64 n) {
  if (n) GTP_LAUNCH(ctx, k_uni_ew, (unsigned)((n + 255) / 256), 256, 0, op, a, a_bcast ? 1 : 0, b, b_bcast ? 1 : 0, r, n);
}

// ---- the Constant/Polynomial dispatch of every op, shared by the gtu_* calls and the program recorder -----------------

UniPlan uni_plan(int op, bool a_const, u64 a_n, bool b_const, u64 b_n) {
  UniPlan p;
  auto ew = [&](bool is_const, u64 n, int e, bool swap, bool a_b, bool b_b) {
    p.is_const = is_const; p.n = is_const ? 1 : n; p.kind = UK_EW; p.ew = e; p.swap = swap; p.a_b = a_b; p.b_b = b_b;
  };
  auto series = [&](bool is_const, u64 n, int kind) { p.is_const = is_const; p.n = is_const ? 1 : n; p.kind = kind; };
  switch (op) {
    case GTU_ADD:
    case GTU_SUB: {   // AddAssign :277-306 / SubAssign :330-362
      const bool sub = op == GTU_SUB;
      if (b_const) ew(a_const, a_n, sub ? UEW_SUB_FIRST : UEW_ADD_FIRST, false, false, true);   // Constant+Constant, or coeffs[0] (+|-)= rhs
      else if (a_const) ew(false, b_n, sub ? UEW_RSUB_FIRST : UEW_ADD_FIRST, true, false, true);   // ws[0] += c  |  ws = -ws; ws[0] += c
      else ew(false, std::min(a_n, b_n), sub ? UEW_SUB : UEW_ADD, false, false, false);   // truncated to the shorter operand (:291, :347)
      break;
    }
    case GTU_MUL:   // :364-389
      if (a_const && b_const) ew(true, 1, UEW_MUL, false, false, false);
      else if (a_const || b_const) ew(false, a_const ? b_n : a_n, UEW_MUL, a_const, false, true);   // coeff *= c
      else series(false, std::min(a_n, b_n), UK_MUL);
      break;
    case GTU_DIV:   // :397-439
      if (a_const && b_const) ew(true, 1, UEW_DIV, false, false, false);
      else if (b_const) ew(false, a_n, UEW_DIV, false, false, true);   // coeff /= c
      else {
        series(false, a_const ? b_n : std::min(a_n, b_n), UK_DIV);
        p.a_b = a_const;
        GTP_CHECK(p.n <= UNI_MAX_DIV, GTP_ERR_ARG, "univariate order > 2048 not supported");
      }
      break;
    case GTU_NEG: ew(a_const, a_n, UEW_NEG, false, false, false); break;   // :308-319
    case GTU_EXP: series(a_const, a_n, a_const ? UK_SCALAR_EXP : UK_EXP); break;   // :151-168
    case GTU_LOG: series(a_const, a_n, a_const ? UK_SCALAR_LOG : UK_LOG); break;   // :170-189
    case GTU_MAX:   // :219-224: constants only
      GTP_CHECK(a_const && b_const, GTP_ERR_INDEX, "Maximum can only be applied to constant Taylor expansions.");
      ew(true, 1, UEW_MAX, false, false, false);
      break;
    default: throw Error(GTP_ERR_ARG, "unknown univariate op");
  }
  return p;
}

void uni_run(Ctx& ctx, const UniPlan& p, const double* a, const double* b, double* r) {
  const double* x = p.swap ? b : a;
  const double* y = p.swap ? a : b;
  switch (p.kind) {
    case UK_EW: uni_ew(ctx, p.ew, x, p.a_b, y, p.b_b, r, p.n); break;
    case UK_MUL: uni_mul(ctx, x, y, r, p.n); break;
    case UK_DIV: uni_div(ctx, x, p.a_b, y, r, p.n); break;
    case UK_EXP: uni_exp(ctx, x, r, p.n); break;
    case UK_LOG: uni_log(ctx, x, r, p.n); break;
    case UK_SCALAR_EXP: launch_scalar_fn(ctx, 0, x, r); break;
    default: launch_scalar_fn(ctx, 1, x, r); break;   // UK_SCALAR_LOG
  }
}

// ---- k_uni_program: a whole recorded program in one CTA ----------------------------------------------------------------
// Instructions are sorted by (level, warp); warp w of level L runs ins[lvl[L * nw + w] .. lvl[L * nw + w + 1]).  A level
// only reads slots of earlier levels, so one __syncthreads() between levels orders every read after its write.  After
// the last level the requested output slots are copied to the gather region, which the host reads back in one copy.
__global__ void __launch_bounds__(1024) k_uni_program(const UniIns* __restrict__ ins, const unsigned* __restrict__ lvl, int nlevels,
                                                      const unsigned* __restrict__ outs, int n_out, double* arena) {
  __shared__ double sh[32][UNI_T / 32];
  const unsigned w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const WarpTeam t{threadIdx.x & 31u};
  for (int L = 0; L < nlevels; L++) {
    const unsigned end = lvl[(u64)L * nw + w + 1];
    for (unsigned i = lvl[(u64)L * nw + w]; i < end; i++) {
      const UniIns in = ins[i];
      const double* x = arena + in.a;
      const double* y = in.b == UNI_NONE ? nullptr : arena + in.b;
      double* r = arena + in.r;
      switch (in.kind) {
        case UK_EW: uni_ew_team(t.lane, 32, in.ew, x, in.a_b, y, in.b_b, r, in.n); break;
        case UK_MUL: uni_mul_team(t.lane, 32, x, y, r, in.n); break;
        case UK_DIV: uni_div_team(t, x, in.a_b, y, r, in.n); break;
        case UK_EXP: uni_exp_team(t, x, r, in.n, sh[w]); break;
        case UK_LOG: uni_log_team(t, x, r, in.n, sh[w]); break;
        case UK_SCALAR_EXP: if (t.lane == 0) r[0] = exp(x[0]); break;   // as k_scalar_fn
        default: if (t.lane == 0) r[0] = log(x[0]); break;              // UK_SCALAR_LOG
      }
      __syncwarp();
    }
    __syncthreads();
  }
  for (int o = 0; o < n_out; o++) {
    const unsigned src = outs[3 * o], len = outs[3 * o + 1], dst = outs[3 * o + 2];
    for (unsigned j = threadIdx.x; j < len; j += blockDim.x) arena[dst + j] = arena[src + j];
  }
}
void uni_program_launch(Ctx& ctx, const UniIns* ins, const unsigned* lvl, int nlevels, int nwarps, const unsigned* outs, int n_out,
                        double* arena) {
  GTP_LAUNCH(ctx, k_uni_program, 1, 32 * nwarps, 0, ins, lvl, nlevels, outs, n_out, arena);
}

// taylor_expansion_of_coeff :78-87
__global__ void k_uni_teoc(const double* __restrict__ in, double* out, u64 n, u64 len) {
  if (threadIdx.x || blockIdx.x) return;
  double factor = 1.0;
  if (len) out[0] = in[n];
  for (u64 k = 1; k < len; k++) {
    factor = __dmul_rn(factor, __ddiv_rn((double)(unsigned)(n + k), (double)(unsigned)k));
    out[k] = __dmul_rn(in[n + k], factor);
  }
}
void uni_teoc(Ctx& ctx, const double* in, double* out, u64 n, u64 len) { GTP_LAUNCH(ctx, k_uni_teoc, 1, 32, 0, in, out, n, len); }

// derivative :47-51 -- factorial(order) * coeffs[order]
__global__ void k_uni_fact(const double* __restrict__ in, u64 order, double* out) {
  if (threadIdx.x || blockIdx.x) return;
  double f = 1.0;
  for (u64 i = 1; i <= order; i++) f = __dmul_rn(f, (double)(unsigned)i);
  out[0] = __dmul_rn(f, in[order]);
}
void uni_factorial_times(Ctx& ctx, const double* in, u64 order, double* out) { GTP_LAUNCH(ctx, k_uni_fact, 1, 32, 0, in, order, out); }

}  // namespace gtp
