// Device-resident N-D recurrences: general power-series division, exp and log of a TaylorPoly
// (multivariate_taylor.rs:1162-1192, :1285-1317, :1335-1386) as ONE cooperative kernel per call.
//
// The reference recursions are forward substitutions.  Unrolled over all axes they read (k, m multi-indices over the
// leading "leaf" axes, rows along the last non-unit axis, (*) the 1-d row convolution):
//
//   div   R[k] = ( X[k] - sum_{m <= k, m != k} R[m] (*) Y[k-m] )  (/)  Y[0]                      (:1170-1191)
//   exp   R[k] = ( sum_{j: j_i = 0 (i < a), 1 <= j_a <= k_a, j_b <= k_b (b > a)} (j_a X[j]) (*) R[k-j] ) / k_a          (:1302-1316)
//   log   Q[k] = ( k_a X[k] - sum_{m: m_i = 0 (i < a), 1 <= m_a < k_a, m_b <= k_b} X[k-m] (*) (m_a R[m])                (:1355-1375)
//                           - sum_{m: m_i = k_i (i <= a), m_b <= k_b, m != k} Q[m] (*) X[0.., k_b-m_b] )  (/)  X[0..0]   (:1376-1383 -> div)
//         R[k] = Q[k] / k_a                                                                                              (:1384)
//
// with a = the first leaf axis on which k is non-zero (the depth at which the reference's recursion reaches row k),
// (/) the 1-d series division along the row, and leaf 0 the 1-d exp_1d / log_1d recurrence.  Every term on the right
// belongs to a leaf of strictly smaller level |m| < |k|, so the leaves of one level |k| are independent: the kernel walks
// the levels with a grid barrier in between -- sum (rs_i - 1) + 1 barriers instead of the host loop of product launches
// (127 / 188 / 527 launches for exp / div / log on 3 x 32; each with a plan build for its ever-changing shapes).
// A work item is (leaf, 32-wide row segment, part of the leaf's pair list); the warps of a CTA split the pairs of a
// part, stage one pair's rows in warp-private shared memory (result rows are read with ld.global.cg: other CTAs wrote
// them in earlier levels) and run a branch-free 32 x 32 DFMA block; partial rows meet in HBM through RED.ADD.F64 and the
// CTA that takes the last ticket of a leaf finalises it (base term, 1-d solve, scaling).
//
// Rounding: this is the reference's recurrence (NOT a reciprocal series), evaluated with FMA and a different summation
// order -- within 1e-12 of the reference on every test input (forward substitution is as well conditioned as the
// reference's own order).  EXACT mode (exp below 2^20 MACs): one warp per (leaf, segment), pairs in the reference's
// order, separate multiply and add, inner row sums from zero -- bit-identical to the reference, like the host loop over
// the reference-order product kernel it replaces.
#include <map>

#include "device_sync.cuh"
#include "kernels.cuh"

namespace gtp {

constexpr int WV_MAXL = 7;      // leaf axes
constexpr int WV_T = 1024;      // threads per CTA: ONE CTA per SM (a grid barrier has at most sm_count arrivals), 32 warps to hide L2 latency
constexpr int WV_W = WV_T / 32;

enum WaveOp : int { WV_DIV = 0, WV_EXP = 1, WV_LOG = 2 };

struct WaveP {
  int nl;                                   // leaf axes
  unsigned rs[WV_MAXL], xs[WV_MAXL], ys[WV_MAXL];
  long long rstr[WV_MAXL], xstr[WV_MAXL], ystr[WV_MAXL];
  unsigned L, xL, yL;                       // row lengths: result, x, y
  unsigned n_leaves, n_levels, nseg, parts;
  const unsigned* leaf_order;               // leaf ids sorted by level
  const unsigned* level_start;              // n_levels + 1
  const double* x;
  const double* y;
  double* r;
  double* q;                                // log: unscaled quotient rows
  double* c;                                // partial right-hand sides (only when a leaf has more than one item)
  unsigned* ticket;                         // per leaf
  unsigned* bar;                            // grid barrier counter (monotonic)
  int has_seed;                             // exp / log: the constant term's exp / log from the host's libm (see kernels.cuh)
  double seed;
  unsigned long long* dbg;                  // GTP_WAVE_DEBUG=1: per-level timestamps of CTA 0 (nullptr otherwise)
};
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// One set of pairs of a leaf: index variables u_i in [lo_i, lo_i + ext_i), first axis slowest.
struct PairSet {
  unsigned lo[WV_MAXL], ext[WV_MAXL];
  long long a_base, b_base;                 // element offsets at u = lo
  long long a_step[WV_MAXL], b_step[WV_MAXL];
  unsigned count;                           // pairs in the set (the excluded last combination already removed)
  int scale_axis;                           // u_{scale_axis} scales the pair (-1: none)
  bool scale_on_a;
  const double* a;                          // rows indexed by j (broadcast side), length aL
  const double* b;                          // rows indexed by t - j, length bL; read with ld.global.cg when b_volatile
  unsigned aL, bL;
  bool b_volatile;
  double sign;
};

struct PairIter {
  unsigned u[WV_MAXL];
  long long ao, bo;
};
__device__ __forceinline__ void pair_seek(const PairSet& s, int nl, unsigned p, PairIter& it) {
  it.ao = s.a_base;
  it.bo = s.b_base;
#pragma unroll
  for (int i = WV_MAXL - 1; i >= 0; --i) {
    if (i < nl) {
      const unsigned q = p / s.ext[i], d = p - q * s.ext[i];
      p = q;
      it.u[i] = s.lo[i] + d;
      it.ao += (long long)d * s.a_step[i];
      it.bo += (long long)d * s.b_step[i];
    }
  }
}
__device__ __forceinline__ void pair_next(const PairSet& s, int nl, PairIter& it) {
#pragma unroll
  for (int i = WV_MAXL - 1; i >= 0; --i) {
    if (i < nl) {
      if (it.u[i] + 1 < s.lo[i] + s.ext[i]) {
        it.u[i]++;
        it.ao += s.a_step[i];
        it.bo += s.b_step[i];
        return;
      }
      const unsigned d = it.u[i] - s.lo[i];
      it.u[i] = s.lo[i];
      it.ao -= (long long)d * s.a_step[i];
      it.bo -= (long long)d * s.b_step[i];
    }
  }
}

// One tile = one pair x one 32-wide chunk jc of the A row: the warp stages A[jc .. jc+31] and the B window
// [t0 - jc - 31, t0 - jc + 31] (zero outside the rows) in its private shared memory and runs a branch-free 32 x 32 block
//     acc(t0 + lane) += sign * A[jc + jj] * B[t0 + lane - jc - jj].
// Tiles are software-pipelined: the global loads of tile i+1 (result rows come from L2: ld.global.cg) are in flight while
// tile i is multiplied.
struct TileRegs { double a, b0, b1; };
__device__ __forceinline__ TileRegs tile_load(const PairSet& s, const PairIter& it, unsigned t0, unsigned jc) {
  const unsigned lane = threadIdx.x & 31u;
  const double* A = s.a + it.ao;
  const double* B = s.b + it.bo;
  double scale = 1.0;
#pragma unroll
  for (int i = 0; i < WV_MAXL; i++)
    if (i == s.scale_axis) scale = (double)it.u[i];
  TileRegs r;
  const unsigned ja = jc + lane;
  r.a = ja < s.aL ? A[ja] : 0.0;
  const long long bi0 = (long long)t0 - (long long)jc - 31 + (long long)lane, bi1 = bi0 + 32;
  r.b0 = (bi0 >= 0 && bi0 < (long long)s.bL) ? (s.b_volatile ? ldcg(B + bi0) : B[bi0]) : 0.0;
  r.b1 = (lane < 31u && bi1 >= 0 && bi1 < (long long)s.bL) ? (s.b_volatile ? ldcg(B + bi1) : B[bi1]) : 0.0;
  if (s.scale_axis >= 0) {
    if (s.scale_on_a) r.a = __dmul_rn(r.a, scale);
    else { r.b0 = __dmul_rn(r.b0, scale); r.b1 = __dmul_rn(r.b1, scale); }
  }
  return r;
}
// range of A chunks whose B window meets [0, bL):  jc in [jc0, j_end) step 32
__device__ __forceinline__ void tile_range(const PairSet& s, unsigned t0, unsigned* jc0, unsigned* j_end) {
  *j_end = min(s.aL, t0 + 32u);
  *jc0 = (t0 + 1u > s.bL + 31u) ? ((t0 - 30u - s.bL) / 32u) * 32u : 0u;
}
// pairs [q0, q1) of set s, row segment t0
template <bool EXACT>
__device__ __forceinline__ void run_pairs(const PairSet& s, int nl, unsigned q0, unsigned q1, unsigned t0, double* sa, double* sb,
                                          double& acc) {
  if (q0 >= q1) return;
  const unsigned lane = threadIdx.x & 31u;
  unsigned jc0, j_end;
  tile_range(s, t0, &jc0, &j_end);
  if (jc0 >= j_end) return;
  PairIter it;
  pair_seek(s, nl, q0, it);
  unsigned q = q0, jc = jc0;
  TileRegs cur = tile_load(s, it, t0, jc);
  double inner = 0.0;
  while (true) {
    sa[lane] = cur.a;
    sb[lane] = cur.b0;
    sb[lane + 32u] = cur.b1;
    __syncwarp();
    const unsigned nj = min(32u, s.aL - jc), jc_now = jc;
    // advance to the next tile and start its loads
    jc += 32u;
    bool pair_done = jc >= j_end, more = true;
    if (pair_done) {
      jc = jc0;
      q++;
      if (q < q1) pair_next(s, nl, it); else more = false;
    }
    if (more) cur = tile_load(s, it, t0, jc);
    if (EXACT) {
      // reference order: j ascending, only the terms that exist (mul_1d :975-979), multiply and add separate;
      // the row sum of one pair starts from zero and is then added (`*z += o`, :998)
      const unsigned t = t0 + lane;
      for (unsigned jj = 0; jj < nj; jj++) {
        const unsigned j = jc_now + jj;
        if (j <= t && t - j < s.bL) inner = __dadd_rn(inner, __dmul_rn(sa[jj], sb[lane + 31u - jj]));
      }
      if (pair_done) {
        acc = __dadd_rn(acc, inner);
        inner = 0.0;
      }
    } else {
      // sa is zero beyond the A row: fixed trip counts (16 or 32), fully unrolled, four independent accumulators
      double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
      const double* sbl = sb + lane + 31u;
#pragma unroll
      for (int jj = 0; jj < 16; jj += 4) {
        c0 = fma(sa[jj], sbl[-jj], c0);
        c1 = fma(sa[jj + 1], sbl[-jj - 1], c1);
        c2 = fma(sa[jj + 2], sbl[-jj - 2], c2);
        c3 = fma(sa[jj + 3], sbl[-jj - 3], c3);
      }
      if (nj > 16u) {
#pragma unroll
        for (int jj = 16; jj < 32; jj += 4) {
          c0 = fma(sa[jj], sbl[-jj], c0);
          c1 = fma(sa[jj + 1], sbl[-jj - 1], c1);
          c2 = fma(sa[jj + 2], sbl[-jj - 2], c2);
          c3 = fma(sa[jj + 3], sbl[-jj - 3], c3);
        }
      }
      acc = fma(s.sign, (c0 + c1) + (c2 + c3), acc);
    }
    __syncwarp();
    if (!more) break;
  }
}

// ---- per-leaf set-up ------------------------------------------------------------------------------------------
template <int OP>
__device__ __forceinline__ int leaf_sets(const WaveP& p, const unsigned* k, PairSet* sets, int* a_out) {
  const int nl = p.nl;
  int a = -1;
  for (int i = 0; i < nl; i++)
    if (k[i] != 0) { a = i; break; }
  *a_out = a;
  if (OP == WV_DIV) {
    PairSet& s = sets[0];
    unsigned cnt = 1;
    s.a_base = s.b_base = 0;
    for (int i = 0; i < nl; i++) {
      const unsigned lo = k[i] + 1 > p.ys[i] ? k[i] + 1 - p.ys[i] : 0;
      s.lo[i] = lo;
      s.ext[i] = k[i] - lo + 1;
      cnt *= s.ext[i];
      s.a_base += (long long)(k[i] - lo) * p.ystr[i];   // Y[k - m]
      s.a_step[i] = -p.ystr[i];
      s.b_base += (long long)lo * p.rstr[i];            // R[m]
      s.b_step[i] = p.rstr[i];
    }
    s.count = cnt - 1;                                  // m = k is the leaf's own 1-d solve
    s.scale_axis = -1;
    s.scale_on_a = false;
    s.a = p.y; s.aL = p.yL;
    s.b = p.r; s.bL = p.L; s.b_volatile = true;
    s.sign = -1.0;
    return 1;
  }
  if (OP == WV_EXP) {
    PairSet& s = sets[0];
    unsigned cnt = 1;
    s.a_base = s.b_base = 0;
    for (int i = 0; i < nl; i++) {
      unsigned lo, ext;
      if (i < a) { lo = 0; ext = 1; }
      else if (i == a) { lo = 1; ext = min(k[i], p.xs[i] - 1); }
      else { lo = 0; ext = min(k[i], p.xs[i] - 1) + 1; }
      s.lo[i] = lo;
      s.ext[i] = ext;
      cnt *= ext;
      s.a_base += (long long)lo * p.xstr[i];            // X[j]
      s.a_step[i] = p.xstr[i];
      s.b_base += (long long)(k[i] - lo) * p.rstr[i];   // R[k - j]
      s.b_step[i] = -p.rstr[i];
    }
    s.count = cnt;
    s.scale_axis = a;
    s.scale_on_a = true;                                // (x * j) * r  (:1306-1309)
    s.a = p.x; s.aL = p.xL;
    s.b = p.r; s.bL = p.L; s.b_volatile = true;
    s.sign = 1.0;
    return 1;
  }
  // WV_LOG: set 0 = the log recurrence, set 1 = the division of the slice by X[0..0, ...]
  {
    PairSet& s = sets[0];
    unsigned cnt = 1;
    bool empty = false;
    s.a_base = s.b_base = 0;
    for (int i = 0; i < nl; i++) {
      unsigned lo, ext;
      if (i < a) { lo = 0; ext = 1; }
      else if (i == a) {
        lo = k[i] + 1 > p.xs[i] ? k[i] + 1 - p.xs[i] : 0;
        if (lo < 1) lo = 1;
        if (lo >= k[i]) { empty = true; ext = 1; } else ext = k[i] - lo;
      } else {
        lo = k[i] + 1 > p.xs[i] ? k[i] + 1 - p.xs[i] : 0;
        ext = k[i] - lo + 1;
      }
      s.lo[i] = lo;
      s.ext[i] = ext;
      cnt *= ext;
      s.a_base += (long long)(k[i] - lo) * p.xstr[i];   // X[k - m]
      s.a_step[i] = -p.xstr[i];
      s.b_base += (long long)lo * p.rstr[i];            // R[m]
      s.b_step[i] = p.rstr[i];
    }
    s.count = empty ? 0 : cnt;
    s.scale_axis = a;
    s.scale_on_a = false;                               // x * (r * j)  (:1361-1365)
    s.a = p.x; s.aL = p.xL;
    s.b = p.r; s.bL = p.L; s.b_volatile = true;
    s.sign = -1.0;
  }
  {
    PairSet& s = sets[1];
    unsigned cnt = 1;
    s.a_base = s.b_base = 0;
    for (int i = 0; i < nl; i++) {
      unsigned lo, ext;
      if (i <= a) { lo = k[i]; ext = 1; }
      else {
        lo = k[i] + 1 > p.xs[i] ? k[i] + 1 - p.xs[i] : 0;
        ext = k[i] - lo + 1;
      }
      s.lo[i] = lo;
      s.ext[i] = ext;
      cnt *= ext;
      if (i > a) s.a_base += (long long)(k[i] - lo) * p.xstr[i];   // X[0.., k_b - m_b]
      s.a_step[i] = i > a ? -p.xstr[i] : 0;
      s.b_base += (long long)lo * p.rstr[i];                        // Q[m]
      s.b_step[i] = p.rstr[i];
    }
    s.count = cnt - 1;
    s.scale_axis = -1;
    s.scale_on_a = false;
    s.a = p.x; s.aL = p.xL;
    s.b = p.q; s.bL = p.L; s.b_volatile = true;
    s.sign = -1.0;
  }
  return 2;
}

__device__ __forceinline__ void decode_leaf(const WaveP& p, unsigned leaf, unsigned* k, long long* roff, long long* xoff, bool* in_x) {
  long long ro = 0, xo = 0;
  bool ok = true;
#pragma unroll
  for (int i = WV_MAXL - 1; i >= 0; --i) {
    if (i < p.nl) {
      const unsigned q = leaf / p.rs[i], d = leaf - q * p.rs[i];
      leaf = q;
      k[i] = d;
      ro += (long long)d * p.rstr[i];
      xo += (long long)d * p.xstr[i];
      ok = ok && d < p.xs[i];
    }
  }
  *roff = ro;
  *xoff = xo;
  *in_x = ok;
}

// 1-d series division along the row, whole CTA:  out[t] = (crow[t] - sum_{s < t, t - s < dl} out[s] * dv[t - s]) / dv[0]
// (right-looking: once out[s] is final every thread retires its term from the pending crow[t]).
__device__ void row_solve(double* crow, const double* __restrict__ dv, unsigned dl, unsigned L) {
  const double d0 = dv[0];
  if (L <= 32u && dl > 1) {
    // short rows: warp 0 alone, the pending row in registers (lane t holds crow[t]), no CTA barriers in the loop
    if (threadIdx.x < 32u) {
      const unsigned lane = threadIdx.x;
      double c = lane < L ? crow[lane] : 0.0;
      const double dvr = lane < dl ? dv[lane] : 0.0;
      const double inv0 = 1.0 / d0;   // one division per row; the product with the reciprocal costs <= 1 ulp per coefficient
      for (unsigned s = 0; s < L; s++) {
        const double rsv = __shfl_sync(0xffffffffu, c, s) * inv0;
        const double dk = __shfl_sync(0xffffffffu, dvr, lane >= s ? lane - s : 0u);
        if (lane == s) c = rsv;
        else if (lane > s) c = fma(-rsv, dk, c);     // dk = 0 beyond the divisor's length
      }
      if (lane < L) crow[lane] = c;
    }
    __syncthreads();
    return;
  }
  if (dl <= 1) {
    for (unsigned t = threadIdx.x; t < L; t += blockDim.x) crow[t] = crow[t] / d0;
    __syncthreads();
    return;
  }
  for (unsigned s = 0; s < L; s++) {
    if (threadIdx.x == 0) crow[s] = crow[s] / d0;
    __syncthreads();
    const double rsv = crow[s];
    const unsigned t_end = min(L, s + dl);
    for (unsigned t = s + 1 + threadIdx.x; t < t_end; t += blockDim.x) crow[t] = fma(-rsv, dv[t - s], crow[t]);
    __syncthreads();
  }
}

// leaf 0 of exp / log: the reference's 1-d recurrences along the row (exp_1d :1271-1283, log_1d :1319-1333), with the
// same split as k_exp_1d / k_log_1d (kernels_rec.cu): short sums by thread 0 in reference order, long ones by the CTA.
__device__ double cta_sum(double v, double* sh) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < WV_W; w++) t += sh[w];
  return t;
}
template <int OP>
__device__ void leaf0_row(const WaveP& p, double* crow, double* red) {
  const unsigned L = p.L, xL = p.xL;
  if (OP == WV_DIV) {
    for (unsigned t = threadIdx.x; t < L; t += blockDim.x) crow[t] = t < xL ? p.x[t] : 0.0;
    __syncthreads();
    row_solve(crow, p.y, p.yL, L);
    for (unsigned t = threadIdx.x; t < L; t += blockDim.x) p.r[t] = crow[t];
    return;
  }
  if (threadIdx.x == 0) crow[0] = p.has_seed ? p.seed : (OP == WV_EXP ? exp(p.x[0]) : log(p.x[0]));
  __syncthreads();
  const double x0 = p.x[0];
  for (unsigned k = 1; k < L; k++) {
    const double kk = (double)k;
    if (OP == WV_EXP) {
      const unsigned hi = xL < k + 1 ? xL : k + 1;
      if (hi <= 32) {
        if (threadIdx.x == 0) {
          double sum = 0.0;
          for (unsigned j = 1; j < hi; j++) sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(p.x[j], (double)j), crow[k - j]));
          crow[k] = __ddiv_rn(sum, kk);
        }
        __syncthreads();
      } else {
        double part = 0.0;
        for (unsigned j = 1 + threadIdx.x; j < hi; j += blockDim.x) part = fma(__dmul_rn(p.x[j], (double)j), crow[k - j], part);
        const double sum = cta_sum(part, red);
        if (threadIdx.x == 0) crow[k] = __ddiv_rn(sum, kk);
        __syncthreads();
      }
    } else {
      unsigned lo = k + 1 > xL ? k + 1 - xL : 0;
      if (lo < 1) lo = 1;
      double sum;
      if (k - lo <= 32) {
        sum = 0.0;
        if (threadIdx.x == 0)
          for (unsigned j = lo; j < k; j++) sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(p.x[k - j], crow[j]), (double)j));
      } else {
        double part = 0.0;
        for (unsigned j = lo + threadIdx.x; j < k; j += blockDim.x) part = fma(p.x[k - j], __dmul_rn(crow[j], (double)j), part);
        sum = cta_sum(part, red);
      }
      if (threadIdx.x == 0) {
        const double xk = k < xL ? p.x[k] : 0.0;
        crow[k] = __ddiv_rn(__ddiv_rn(__dsub_rn(__dmul_rn(xk, kk), sum), x0), kk);
      }
      __syncthreads();
    }
  }
  for (unsigned t = threadIdx.x; t < L; t += blockDim.x) p.r[t] = crow[t];
  // (log: leaf 0 has no quotient row -- no other leaf reads Q[0])
}

// ---- the kernel -------------------------------------------------------------------------------------------------
// dynamic shared memory: crow[Lpad] | stage: WV_W x (32 + 64) | red[WV_W x 32]
template <int OP, bool EXACT>
__global__ void __launch_bounds__(WV_T) k_rec_wave(const WaveP p) {
  extern __shared__ __align__(16) double wsm[];
  const unsigned Lpad = (p.L + 31u) & ~31u;
  double* crow = wsm;
  double* stage = wsm + Lpad;
  double* red = stage + WV_W * 96;
  __shared__ unsigned s_last;
  // leaf descriptors are built once per item (thread 0 of the CTA; lane 0 of the warp in EXACT mode) and read by everyone
  __shared__ PairSet s_sets[EXACT ? WV_W : 1][2];
  __shared__ unsigned s_k[EXACT ? WV_W : 1][WV_MAXL];
  __shared__ long long s_off[EXACT ? WV_W : 1][2];
  __shared__ int s_misc[EXACT ? WV_W : 1][3];   // a, nsets, in_x
  const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  double* sa = stage + w * 96;
  double* sb = sa + 32;
  unsigned phase = 0;

  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[0] = gtimer();
  if (blockIdx.x == 0) leaf0_row<OP>(p, crow, red);
  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[1] = gtimer();
  grid_barrier(p.bar, phase);
  if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[2] = gtimer();

  for (unsigned level = 1; level < p.n_levels; level++) {
    const unsigned l0 = p.level_start[level], l1 = p.level_start[level + 1];
    // parts per leaf adapt to the level: narrow levels (few leaves -- but on the late ones each leaf has the most pairs)
    // are split over the whole grid, wide levels take one CTA per (leaf, segment) and skip the atomics
    const unsigned parts = EXACT ? 1u : max(1u, min(p.parts, gridDim.x / max(1u, (l1 - l0) * p.nseg)));
    const unsigned per_leaf = p.nseg * parts;
    if (EXACT) {
      // one warp per (leaf, segment): pairs in reference order, element-wise finalisation (exp only)
      const unsigned items = (l1 - l0) * p.nseg;
      for (unsigned item = blockIdx.x * WV_W + w; item < items; item += gridDim.x * WV_W) {
        const unsigned leaf = p.leaf_order[l0 + item / p.nseg], seg = item % p.nseg;
        __syncwarp();
        if (lane == 0) {
          unsigned k[WV_MAXL];
          long long roff, xoff;
          bool in_x;
          int a;
          decode_leaf(p, leaf, k, &roff, &xoff, &in_x);
          leaf_sets<OP>(p, k, s_sets[w], &a);
          s_off[w][0] = roff;
          s_misc[w][0] = (int)k[a];
        }
        __syncwarp();
        const long long roff = s_off[w][0];
        const unsigned ka_u = (unsigned)s_misc[w][0];
        double total = 0.0;
        run_pairs<true>(s_sets[w][0], p.nl, 0, s_sets[w][0].count, seg * 32u, sa, sb, total);
        const unsigned t = seg * 32u + lane;
        if (t < p.L) p.r[roff + t] = __ddiv_rn(total, (double)ka_u);
      }
    } else {
      const unsigned items = (l1 - l0) * per_leaf;
      for (unsigned item = blockIdx.x; item < items; item += gridDim.x) {
        const unsigned leaf = p.leaf_order[l0 + item / per_leaf];
        const unsigned sub = item % per_leaf, seg = sub / parts, part = sub % parts;
        if (threadIdx.x == 0) {
          unsigned k[WV_MAXL];
          long long roff, xoff;
          bool in_x;
          int a;
          decode_leaf(p, leaf, k, &roff, &xoff, &in_x);
          s_misc[0][1] = leaf_sets<OP>(p, k, s_sets[0], &a);
          s_off[0][0] = roff;
          s_off[0][1] = xoff;
          s_misc[0][0] = (int)k[a];
          s_misc[0][2] = in_x ? 1 : 0;
        }
        __syncthreads();
        const PairSet* sets = s_sets[0];
        const long long roff = s_off[0][0], xoff = s_off[0][1];
        const int nsets = s_misc[0][1];
        const bool in_x = s_misc[0][2] != 0;
        const double ka = (double)s_misc[0][0];
        unsigned total_pairs = 0;
        for (int si = 0; si < nsets; si++) total_pairs += sets[si].count;
        // A leaf with few pairs is not split (every CTA of the leaf derives the same count): its one CTA per segment skips
        // the atomics and the ticket, which cost more than two pairs per warp.
        const unsigned parts_leaf = max(1u, min(parts, total_pairs / (2u * WV_W)));
        const unsigned per_leaf_now = p.nseg * parts_leaf;
        if (part >= parts_leaf) { __syncthreads(); continue; }
        // contiguous share of the pair list for warp (part, w)
        const unsigned nshare = parts_leaf * WV_W, me = part * WV_W + w;
        const unsigned chunk = (total_pairs + nshare - 1) / nshare;
        unsigned q0 = min(total_pairs, me * chunk), q1 = min(total_pairs, q0 + chunk);
        double acc = 0.0;
        unsigned base = 0;
        for (int si = 0; si < nsets; si++) {
          const unsigned cnt = sets[si].count;
          const unsigned b0 = max(q0, base), b1 = min(q1, base + cnt);
          if (b0 < b1) run_pairs<false>(sets[si], p.nl, b0 - base, b1 - base, seg * 32u, sa, sb, acc);
          base += cnt;
        }
        // the CTA's partial row segment
        red[w * 32 + lane] = acc;
        __syncthreads();
        if (w == 0) {
          double v = 0.0;
#pragma unroll
          for (int ww = 0; ww < WV_W; ww++) v += red[ww * 32 + lane];
          const unsigned t = seg * 32u + lane;
          if (per_leaf_now == 1) crow[lane] = v;
          else if (t < p.L) atomicAdd(p.c + (size_t)leaf * p.L + t, v);
        }
        bool last = true;
        if (per_leaf_now > 1) {
          __syncthreads();
          if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(p.ticket + leaf, 1u) == per_leaf_now - 1 ? 1u : 0u;
            __threadfence();
          }
          __syncthreads();
          last = s_last != 0;
          if (last)
            for (unsigned t = threadIdx.x; t < p.L; t += blockDim.x) crow[t] = ldcg(p.c + (size_t)leaf * p.L + t);
        }
        __syncthreads();
        if (last) {
          // base term, solve, scaling
          if (OP == WV_DIV || OP == WV_LOG) {
            for (unsigned t = threadIdx.x; t < p.L; t += blockDim.x) {
              double xv = (in_x && t < p.xL) ? p.x[xoff + t] : 0.0;
              if (OP == WV_LOG) xv = __dmul_rn(ka, xv);
              crow[t] = xv + crow[t];
            }
            __syncthreads();
            row_solve(crow, OP == WV_DIV ? p.y : p.x, OP == WV_DIV ? p.yL : p.xL, p.L);
            for (unsigned t = threadIdx.x; t < p.L; t += blockDim.x) {
              if (OP == WV_LOG) {
                p.q[roff + t] = crow[t];
                p.r[roff + t] = crow[t] / ka;
              } else {
                p.r[roff + t] = crow[t];
              }
            }
          } else {
            for (unsigned t = threadIdx.x; t < p.L; t += blockDim.x) p.r[roff + t] = crow[t] / ka;
          }
        }
        __syncthreads();
      }
    }
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[2 * level + 1] = gtimer();   // work of the level done (CTA 0)
    grid_barrier(p.bar, phase);
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[2 * level + 2] = gtimer();   // barrier passed
  }
}

// ---- host ---------------------------------------------------------------------------------------------------------
struct WaveTables {
  BufP order, start;
  unsigned n_leaves = 0, n_levels = 0, widest = 0;
};
using WaveCache = std::map<std::vector<u64>, std::shared_ptr<WaveTables>>;

static std::shared_ptr<WaveTables> wave_tables(Ctx& ctx, const std::vector<u64>& leaf_ext) {
  if (!ctx.wave_tables) ctx.wave_tables = std::make_shared<WaveCache>();
  auto& cache = *std::static_pointer_cast<WaveCache>(ctx.wave_tables);
  auto it = cache.find(leaf_ext);
  if (it != cache.end()) return it->second;
  auto t = std::make_shared<WaveTables>();
  u64 n = 1, levels = 1;
  for (u64 e : leaf_ext) { n *= e; levels += e - 1; }
  t->n_leaves = (unsigned)n;
  t->n_levels = (unsigned)levels;
  std::vector<unsigned> lvl(n), start(levels + 1, 0), order(n);
  {
    std::vector<unsigned> k(leaf_ext.size(), 0);
    unsigned s = 0;
    for (u64 leaf = 0; leaf < n; leaf++) {
      lvl[leaf] = s;
      start[s + 1]++;
      for (int i = (int)leaf_ext.size() - 1; i >= 0; --i) {   // odometer, last axis fastest (row-major leaf ids)
        if (k[i] + 1 < leaf_ext[i]) { k[i]++; s++; break; }
        s -= k[i];
        k[i] = 0;
      }
    }
  }
  for (u64 l = 0; l < levels; l++) {
    t->widest = std::max(t->widest, start[l + 1]);
    start[l + 1] += start[l];
  }
  {
    std::vector<unsigned> fill(start.begin(), start.end() - 1);
    for (u64 leaf = 0; leaf < n; leaf++) order[fill[lvl[leaf]]++] = (unsigned)leaf;
  }
  t->order = ctx.alloc((n + 1) / 2 + 1);
  t->start = ctx.alloc((levels + 2) / 2 + 1);
  GTP_CUDA(cudaMemcpyAsync(t->order->d, order.data(), n * sizeof(unsigned), cudaMemcpyHostToDevice, ctx.stream));
  GTP_CUDA(cudaMemcpyAsync(t->start->d, start.data(), (levels + 1) * sizeof(unsigned), cudaMemcpyHostToDevice, ctx.stream));
  if (cache.size() > 32) cache.clear();
  cache[leaf_ext] = t;
  return t;
}

template <int OP, bool EXACT>
static bool wave_launch(Ctx& ctx, WaveP& p, unsigned want_ctas, size_t smem) {
  static int coop[64] = {};           // 0 unknown, 1 yes, -1 no
  int& c = coop[ctx.device & 63];
  if (c == 0) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, ctx.device);
    c = v ? 1 : -1;
  }
  if (c < 0) return false;
  auto* fn = k_rec_wave<OP, EXACT>;
  allow_dyn_smem(fn, ctx.device, smem);   // static + dynamic may pass 48 KB
  int per_sm = 0;
  GTP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, WV_T, smem));
  if (per_sm < 1) return false;
  const unsigned max_ctas = (unsigned)ctx.sm_count;
  const unsigned grid = std::max(1u, std::min(want_ctas, max_ctas));
  void* args[] = {(void*)&p};
  const double t0 = ctx.hist ? Ctx::now() : 0.0;
  GTP_CUDA(cudaLaunchCooperativeKernel((const void*)fn, dim3(grid), dim3(WV_T), args, smem, ctx.stream));
  ctx.launches++;
  if (ctx.hist) {
    (*ctx.hist)[EXACT ? "k_rec_wave<exact>" : "k_rec_wave"]++;
    ctx.t_launch += Ctx::now() - t0;
  }
  return true;
}

// Returns false when the shapes are outside this kernel's domain (the caller keeps its host-loop path).
// op: 0 div (y = divisor), 1 exp, 2 log.  All shapes have the same ndim; r is dense over rs and fully overwritten.
bool launch_rec_wave(Ctx& ctx, int op, const double* x, const Shape& xs, const double* y, const Shape& ys, double* r,
                     const Shape& rs, bool exact, const double* seed) {
  const int nd = (int)rs.size();
  std::vector<int> eff;
  for (int d = 0; d < nd; d++) {
    if (rs[d] == 1) {
      if (xs[d] != 1 || (op == WV_DIV && ys[d] != 1)) return false;
      continue;
    }
    eff.push_back(d);
  }
  if (eff.size() < 2 || eff.size() > (size_t)WV_MAXL + 1) return false;
  if (prod(rs) >= (1ull << 31) || prod(xs) >= (1ull << 31)) return false;
  Shape xst(nd, 1), yst(nd, 1), rst(nd, 1);
  for (int i = nd - 2; i >= 0; --i) {
    xst[i] = xst[i + 1] * xs[i + 1];
    rst[i] = rst[i + 1] * rs[i + 1];
    if (op == WV_DIV) yst[i] = yst[i + 1] * ys[i + 1];
  }
  WaveP p;
  memset(&p, 0, sizeof(p));
  const int nl = (int)eff.size() - 1, row = eff.back();
  if (rst[row] != 1 || (xs[row] > 1 && xst[row] != 1) || (op == WV_DIV && ys[row] > 1 && yst[row] != 1)) return false;
  p.nl = nl;
  std::vector<u64> leaf_ext;
  for (int i = 0; i < nl; i++) {
    const int d = eff[i];
    if (op != WV_DIV && xs[d] < 2) return false;   // exp / log: x is non-constant wherever the result is
    p.rs[i] = (unsigned)rs[d];
    p.xs[i] = (unsigned)xs[d];
    p.ys[i] = op == WV_DIV ? (unsigned)ys[d] : 1u;
    p.rstr[i] = (long long)rst[d];
    p.xstr[i] = (long long)xst[d];
    p.ystr[i] = op == WV_DIV ? (long long)yst[d] : 0;
    leaf_ext.push_back(rs[d]);
  }
  p.L = (unsigned)rs[row];
  p.xL = (unsigned)xs[row];
  p.yL = op == WV_DIV ? (unsigned)ys[row] : 1u;
  if (op != WV_DIV && p.xL < 2) return false;
  const unsigned Lpad = (p.L + 31u) & ~31u;
  const size_t smem = ((size_t)Lpad + WV_W * 96 + WV_W * 32) * sizeof(double);
  if (smem > 200 * 1024) return false;
  if (exact && op != WV_EXP) return false;
  auto tab = wave_tables(ctx, leaf_ext);
  p.n_leaves = tab->n_leaves;
  p.n_levels = tab->n_levels;
  p.leaf_order = reinterpret_cast<const unsigned*>(tab->order->d);
  p.level_start = reinterpret_cast<const unsigned*>(tab->start->d);
  p.nseg = Lpad / 32;
  const unsigned max_grid = (unsigned)ctx.sm_count;   // one 512-thread CTA per SM
  unsigned want;
  if (exact) {
    p.parts = 1;
    want = (tab->widest * p.nseg + WV_W - 1) / WV_W;
  } else {
    // p.parts is the CAP on the parts per leaf (the kernel picks min(cap, grid / items of the level) per level): no more
    // parts than the largest leaf has pairs for its warps
    u64 pairs_max = 1;
    for (int i = 0; i < nl; i++) pairs_max *= std::max<u64>(1, std::min<u64>(p.rs[i], op == WV_DIV ? p.ys[i] : p.xs[i]));
    p.parts = (unsigned)std::max<u64>(1, std::min<u64>(max_grid, pairs_max / (2 * WV_W)));
    want = (unsigned)std::min<u64>((u64)tab->widest * p.nseg * p.parts, max_grid);
  }
  p.x = x;
  p.y = y;
  p.r = r;
  p.has_seed = seed ? 1 : 0;
  p.seed = seed ? *seed : 0.0;
  // scratch: barrier counter | tickets | partial rows | quotient rows
  const bool multi = !exact && (p.nseg > 1 || p.parts > 1);
  const u64 n_out = (u64)p.n_leaves * p.L;
  const u64 head = 2 + (multi ? (p.n_leaves + 1) / 2 : 0);
  BufP scratch = ctx.alloc(head + (multi ? n_out : 0) + (op == WV_LOG ? n_out : 0));
  GTP_CUDA(cudaMemsetAsync(scratch->d, 0, (head + (multi ? n_out : 0)) * sizeof(double), ctx.stream));
  p.bar = reinterpret_cast<unsigned*>(scratch->d);
  p.ticket = reinterpret_cast<unsigned*>(scratch->d + 2);
  p.c = scratch->d + head;
  p.q = scratch->d + head + (multi ? n_out : 0);
  static const bool debug = getenv("GTP_WAVE_DEBUG") && getenv("GTP_WAVE_DEBUG")[0] == '1';
  BufP dbg;
  if (debug) {
    dbg = ctx.alloc(2 * (u64)p.n_levels + 4);
    GTP_CUDA(cudaMemsetAsync(dbg->d, 0, (2 * (u64)p.n_levels + 4) * 8, ctx.stream));
    p.dbg = reinterpret_cast<unsigned long long*>(dbg->d);
  }
  bool ok;
  if (op == WV_DIV) ok = wave_launch<WV_DIV, false>(ctx, p, want, smem);
  else if (op == WV_EXP) ok = exact ? wave_launch<WV_EXP, true>(ctx, p, want, smem) : wave_launch<WV_EXP, false>(ctx, p, want, smem);
  else ok = wave_launch<WV_LOG, false>(ctx, p, want, smem);
  if (debug && ok) {
    std::vector<unsigned long long> h(2 * (size_t)p.n_levels + 4);
    GTP_CUDA(cudaMemcpyAsync(h.data(), dbg->d, h.size() * 8, cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    fprintf(stderr, "[wave op %d] leaves %u levels %u nseg %u parts %u exact %d: leaf0 %.1f us, barrier0 %.1f us\n", op, p.n_leaves, p.n_levels,
            p.nseg, p.parts, (int)exact, (h[1] - h[0]) * 1e-3, (h[2] - h[1]) * 1e-3);
    double work = 0, bar = 0;
    for (unsigned l = 1; l < p.n_levels; l++) {
      work += (h[2 * l + 1] - h[2 * l]) * 1e-3;
      bar += (h[2 * l + 2] - h[2 * l + 1]) * 1e-3;
      if (l <= 3 || l % 8 == 0) fprintf(stderr, "   level %u: work(CTA0) %.2f us, wait+barrier %.2f us\n", l, (h[2 * l + 1] - h[2 * l]) * 1e-3, (h[2 * l + 2] - h[2 * l + 1]) * 1e-3);
    }
    fprintf(stderr, "   total %.1f us: CTA0 work %.1f us, CTA0 wait+barrier %.1f us\n", (h[2 * p.n_levels] - h[0]) * 1e-3, work, bar);
  }
  return ok;
}

}  // namespace gtp
