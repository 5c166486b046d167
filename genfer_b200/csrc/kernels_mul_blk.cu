// Generic 2x2-blocked, chunk-aware DFMA kernel for the truncated N-D product
// (multivariate_taylor.rs:984-1012) on dense operands whose last axis has the same length in X, Y and Z.
//
//   axes = [ A-axes ... | b1 | b2 | L ],   L = Lc chunks of LT doubles (LT in {8,10,12,14,16}, Lc >= 1)
//
// * One thread multiplies TWO adjacent x rows (j1; a, a+1; chunk jc) with TWO adjacent y rows
//   (m1; b, b+1; chunk mc) -- a, b even -- and accumulates the four row convolutions into the THREE
//   output rows (j1+m1; s, s+1, s+2; chunk kc), s = a+b, that it keeps in registers.  The row
//   convolution comes in two kinds because the last axis is chunked:
//       lo:  z[k] += sum_{j<=k} x[j] * y[k-j]          (jc + mc     == kc)   LT(LT+1)/2 DFMA
//       hi:  z[k] += sum_{j> k} x[j] * y[LT+k-j]       (jc + mc + 1 == kc)   LT(LT-1)/2 DFMA
//   Both are fully unrolled with exact trip counts: no padded multiply-adds except the rows that fall
//   outside the truncation at an odd/last row pair (those x/y rows are zero-filled in shared memory
//   or the z row is dropped at the flush).
// * A slab = the (b1, b2, L) sub-tensor at one A index (b1 may be folded into the A axes when the slab
//   would not fit).  G slab pairs (X[jA], Y[kA-jA]) of one output slab kA are staged per round with
//   cp.async; the items of a round -- (z row block, x row pair, y row pair, kind, g) -- come from a
//   host-built table that deals them EVENLY to the threads, ordered by z row block so a thread flushes
//   (RED.ADD.F64 to HBM) only when its block changes.
// * A-axes: work unit = (output slab kA, chunk [q0,q1) of the jA box), longest first (LPT).
#include "kernels.cuh"

namespace gtp {

constexpr int BT = 128;       // threads per CTA
constexpr int B_MAXA = 6;
constexpr int B_MAXG = 8;

struct BlkP {
  int na;
  unsigned xa[B_MAXA], ya[B_MAXA], ra[B_MAXA];
  long long xastr[B_MAXA], yastr[B_MAXA];
  unsigned rows_a0;
  // global slab geometry (rows of LT doubles): plane = b2*Lc rows
  unsigned x_planes, x_prow, y_planes, y_prow;   // planes (b1) and rows per plane (b2*Lc) in X / Y
  unsigned z_rows;                               // rows per output slab
  unsigned z_pair_stride;                        // Lc of the result: rows between (s) and (s+1)
  // shared-memory geometry (doubles)
  unsigned x_plane_sm, y_plane_sm;               // padded plane strides
  unsigned x_slab_sm, y_slab_sm;                 // per staged slab
  unsigned x_pair_off, y_pair_off;               // distance between the two rows of a pair (Lc*ROW)
  int G;
  int nsteps_lo, nsteps;   // steps [0, nsteps_lo) hold `lo` items, [nsteps_lo, nsteps) `hi` items
  const uint2* table;    // [nsteps][BT]
  const uint4* units;    // {packed kA index, q0, q1, k along A axis 0}
  const double* x;
  const double* y;
  double* out;
};

// table entry: .x = xoff (20) | g << 20 (4) | kind << 24 | z1 valid << 25 | z2 valid << 26 | valid << 31
//              .y = yoff (20) | zrow << 20 (12)
constexpr unsigned BE_VALID = 1u << 31;

template <int LT> struct BRow { static constexpr int value = ((LT / 2) % 2 == 1) ? LT : LT + 2; };

template <int LT>
__device__ __forceinline__ void blk_flush(double (&z)[LT], double* __restrict__ dst, bool write) {
#pragma unroll
  for (int i = 0; i < LT; i++) {
    if (write) atomicAdd(dst + i, z[i]);
    z[i] = 0.0;
  }
}

template <int LT, bool HI>
__device__ __forceinline__ void blk_item(double (&z0)[LT], double (&z1)[LT], double (&z2)[LT], const double* __restrict__ xs,
                                         const double* __restrict__ xs2, const double* __restrict__ ys,
                                         const double* __restrict__ ys2) {
  double y0[LT], y1[LT];
#pragma unroll
  for (int i = 0; i < LT; i += 2) {
    double2 u = *reinterpret_cast<const double2*>(ys + i);
    double2 v = *reinterpret_cast<const double2*>(ys2 + i);
    y0[i] = u.x; y0[i + 1] = u.y;
    y1[i] = v.x; y1[i + 1] = v.y;
  }
#pragma unroll
  for (int j = 0; j < LT; j += 2) {
    double2 xa = *reinterpret_cast<const double2*>(xs + j);
    double2 xb = *reinterpret_cast<const double2*>(xs2 + j);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const double xaj = h ? xa.y : xa.x, xbj = h ? xb.y : xb.x;
      const int jj = j + h;
      if (!HI) {
#pragma unroll
        for (int kk = jj; kk < LT; kk++) {
          z0[kk] = fma(xaj, y0[kk - jj], z0[kk]);
          z1[kk] = fma(xaj, y1[kk - jj], z1[kk]);
          z1[kk] = fma(xbj, y0[kk - jj], z1[kk]);
          z2[kk] = fma(xbj, y1[kk - jj], z2[kk]);
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < jj; kk++) {
          z0[kk] = fma(xaj, y0[LT + kk - jj], z0[kk]);
          z1[kk] = fma(xaj, y1[LT + kk - jj], z1[kk]);
          z1[kk] = fma(xbj, y0[LT + kk - jj], z1[kk]);
          z2[kk] = fma(xbj, y1[LT + kk - jj], z2[kk]);
        }
      }
    }
  }
}

template <int LT, bool CHUNKED>
__global__ void __launch_bounds__(BT) k_mul_blk(const BlkP p) {
  constexpr int ROW = BRow<LT>::value;
  constexpr int V2 = LT / 2;
  extern __shared__ __align__(16) double smem[];
  double* Xs = smem;
  double* Ys = smem + (size_t)p.G * p.x_slab_sm;
  const int tid = threadIdx.x;
  const int bt = blockDim.x;
  const uint4 unit = p.units[blockIdx.x];

  // zero the whole staging area once: padding rows (odd b2) must read as zeros forever
  {
    const int total = p.G * (int)(p.x_slab_sm + p.y_slab_sm);
    for (int i = tid * 2; i < total; i += bt * 2) *reinterpret_cast<double2*>(smem + i) = make_double2(0.0, 0.0);
  }

  unsigned k[B_MAXA], lo[B_MAXA], ext[B_MAXA];
  {
    unsigned rem = unit.x;
#pragma unroll
    for (int a = B_MAXA - 1; a >= 0; --a) {
      if (a < p.na) {
        unsigned len = (a == 0) ? p.rows_a0 : p.ra[a];
        unsigned idx = rem % len;
        rem /= len;
        k[a] = (a == 0) ? unit.w : idx;
        unsigned l = (k[a] + 1 > p.ya[a]) ? k[a] + 1 - p.ya[a] : 0;
        unsigned h = (k[a] + 1 < p.xa[a]) ? k[a] + 1 : p.xa[a];
        lo[a] = l;
        ext[a] = h > l ? h - l : 0;
      } else {
        k[a] = lo[a] = 0;
        ext[a] = 1;
      }
    }
  }
  double* out_slab = p.out + (size_t)unit.x * p.z_rows * LT;

  double z0[LT], z1[LT], z2[LT];
#pragma unroll
  for (int i = 0; i < LT; i++) z0[i] = z1[i] = z2[i] = 0.0;
  unsigned cur = 0xffffffffu;   // (zrow << 2 | valid flags) of the block held in z0..z2
  unsigned round = 0;

  for (unsigned q = unit.y; q < unit.z; q += p.G, ++round) {
    const int ng = min((unsigned)p.G, unit.z - q);
    __syncthreads();  // everyone is done with the previous round's slabs (and with the zero fill)
    for (int g = 0; g < ng; g++) {
      long long xo = 0, yo = 0;
      unsigned rem = q + g;
#pragma unroll
      for (int a = B_MAXA - 1; a >= 0; --a) {
        if (a < p.na) {
          unsigned j = lo[a] + rem % ext[a];
          rem /= ext[a];
          xo += (long long)j * p.xastr[a];
          yo += (long long)(k[a] - j) * p.yastr[a];
        }
      }
      const double2* gx = reinterpret_cast<const double2*>(p.x + xo);
      const double2* gy = reinterpret_cast<const double2*>(p.y + yo);
      double* xs = Xs + (size_t)g * p.x_slab_sm;
      double* ys = Ys + (size_t)g * p.y_slab_sm;
      const int nx = (int)(p.x_planes * p.x_prow) * V2, ny = (int)(p.y_planes * p.y_prow) * V2;
      for (int i = tid; i < nx; i += bt) {
        int r = i / V2, c = i - r * V2;
        int pl = r / (int)p.x_prow, rr = r - pl * (int)p.x_prow;
        cp_async16(xs + pl * p.x_plane_sm + rr * ROW + 2 * c, gx + i);
      }
      for (int i = tid; i < ny; i += bt) {
        int r = i / V2, c = i - r * V2;
        int pl = r / (int)p.y_prow, rr = r - pl * (int)p.y_prow;
        cp_async16(ys + pl * p.y_plane_sm + rr * ROW + 2 * c, gy + i);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    // Two phases per round -- all `lo` items, then all `hi` items -- so that every thread of a warp runs the
    // same unrolled body at the same step (no divergence).  The walk direction alternates between rounds so
    // the z row block at the seam stays in registers.
    const bool fwd = (round & 1u) == 0;
#pragma unroll
    for (int ph = 0; ph < (CHUNKED ? 2 : 1); ph++) {
      const bool hi = CHUNKED && (fwd ? ph == 1 : ph == 0);
      const int s_begin = hi ? p.nsteps_lo : 0, s_end = hi ? p.nsteps : p.nsteps_lo;
      const int cnt = s_end - s_begin;
      if (cnt <= 0) continue;
      int step = fwd ? s_begin : s_end - 1;
      const int dstep = fwd ? 1 : -1;
      uint2 e = p.table[step * bt + tid];
      for (int s = 0; s < cnt; ++s) {
        step += dstep;
        uint2 en = make_uint2(0u, 0u);
        if (s + 1 < cnt) en = p.table[step * bt + tid];
        if ((e.x & BE_VALID) && (int)((e.x >> 20) & 15u) < ng) {
          const unsigned zkey = ((e.y >> 20) << 2) | ((e.x >> 25) & 3u);
          if (zkey != cur) {
            if (cur != 0xffffffffu) {
              double* dst = out_slab + (size_t)(cur >> 2) * LT;
              blk_flush<LT>(z0, dst, true);
              blk_flush<LT>(z1, dst + (size_t)p.z_pair_stride * LT, (cur & 1u) != 0);
              blk_flush<LT>(z2, dst + (size_t)2 * p.z_pair_stride * LT, (cur & 2u) != 0);
            }
            cur = zkey;
          }
          const double* xs = Xs + (e.x & 0xfffffu);
          const double* ys = Ys + (e.y & 0xfffffu);
          if (hi) blk_item<LT, true>(z0, z1, z2, xs, xs + p.x_pair_off, ys, ys + p.y_pair_off);
          else blk_item<LT, false>(z0, z1, z2, xs, xs + p.x_pair_off, ys, ys + p.y_pair_off);
        }
        e = en;
      }
    }
  }
  if (cur != 0xffffffffu) {
    double* dst = out_slab + (size_t)(cur >> 2) * LT;
    blk_flush<LT>(z0, dst, true);
    blk_flush<LT>(z1, dst + (size_t)p.z_pair_stride * LT, (cur & 1u) != 0);
    blk_flush<LT>(z2, dst + (size_t)2 * p.z_pair_stride * LT, (cur & 2u) != 0);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct BlkGeom {
  int nd, na;          // na = number of A axes (b1 folded in when fold_b1)
  bool fold_b1;        // the slab is (b2, L) only
  u64 lt, lc;          // chunk length, chunks per row
  u64 xb1, xb2, yb1, yb2, rb1, rb2;   // slab plane counts (b1 = 1 when folded) and rows
  u64 row;             // padded row length in smem (doubles)
  u64 xplane, yplane, xslab, yslab;   // smem strides (doubles)
  int G;
  size_t smem;
};

struct BlkGeom;
static bool blk_dense(const BlkGeom& g);

static bool blk_geom(const MulArgs& a, BlkGeom* g) {
  const int nd = a.ndim;
  if (nd < 3) return false;
  const u64 ltt = a.rs[nd - 1];
  if (a.xs[nd - 1] != ltt || a.ys[nd - 1] != ltt) return false;
  const u64 lt = dfma_chunk(ltt);
  if (!lt) return false;
  for (int d = 0; d < nd; d++)
    if (a.xs[d] == 0 || a.ys[d] == 0 || a.rs[d] == 0) return false;
  g->nd = nd;
  g->lt = lt;
  g->lc = ltt / lt;
  g->row = ((lt / 2) % 2 == 1) ? lt : lt + 2;
  g->xb2 = a.xs[nd - 2]; g->yb2 = a.ys[nd - 2]; g->rb2 = a.rs[nd - 2];
  auto layout = [&](u64 xb1, u64 yb1) {
    u64 xrows = ((g->xb2 + 1) / 2 * 2) * g->lc, yrows = ((g->yb2 + 1) / 2 * 2) * g->lc;
    g->xplane = xrows * g->row + 2;   // +2 doubles: consecutive planes start in different 16-byte bank groups
    g->yplane = yrows * g->row + 2;
    // staged slabs g = 0..G-1 start in different 16-byte bank groups: slab stride = odd number of groups
    g->xslab = odd_groups(xb1 * g->xplane + 2);
    g->yslab = odd_groups(yb1 * g->yplane + 2);
  };
  // try the 3-axis slab first
  const size_t budget = 100 * 1024;   // two CTAs per SM
  g->fold_b1 = true;
  if (nd >= 4) {
    layout(a.xs[nd - 3], a.ys[nd - 3]);
    if ((g->xslab + g->yslab) * 8 <= budget && a.rs[nd - 3] * a.rs[nd - 2] * g->lc < 4096) g->fold_b1 = false;
  }
  if (g->fold_b1) {
    g->xb1 = g->yb1 = g->rb1 = 1;
    g->na = nd - 2;
    layout(1, 1);
  } else {
    g->xb1 = a.xs[nd - 3]; g->yb1 = a.ys[nd - 3]; g->rb1 = a.rs[nd - 3];
    g->na = nd - 3;
  }
  if (g->na < 1 || g->na > B_MAXA) return false;
  if (g->rb1 * g->rb2 * g->lc >= 4096) return false;
  const u64 pair = (g->xslab + g->yslab) * 8;
  if (pair > budget) return false;
  g->G = (int)std::max<u64>(1, std::min<u64>(B_MAXG, budget / pair));
  if (g->G * std::max(g->xslab, g->yslab) >= (1u << 20)) return false;
  g->smem = (size_t)g->G * pair;
  return true;
}

bool blk_mul_applicable(const Ctx& ctx, const MulArgs& a) {
  BlkGeom g;
  if (a.accumulate) return false;
  if (!blk_geom(a, &g)) return false;
  u64 slabs = a.row_count;
  for (int d = 1; d < g.na; d++) slabs *= a.rs[d];
  return slabs >= 64 || (slabs >= 1 && (ctx.fast_mul == 2 || args_macs(a) >= DFMA_MIN_MACS));   // mode 2 forces the kernel (tests)
}

struct BlkItem { unsigned xoff, yoff, zrow, kind, zv; };

// Items of ONE slab pair, grouped by z row block (k1, sp, kc); see the header comment.
static void build_items(const BlkGeom& g, std::vector<std::vector<BlkItem>>* blocks) {
  const u64 nxp = (g.xb2 + 1) / 2, nyp = (g.yb2 + 1) / 2, nzp = (g.rb2 + 1) / 2;
  for (u64 k1 = 0; k1 < g.rb1; k1++) {
    const u64 lo1 = sat_sub(k1 + 1, g.yb1), hi1 = std::min(k1 + 1, g.xb1);
    for (u64 sp = 0; sp < nzp; sp++)
      for (u64 kc = 0; kc < g.lc; kc++) {
        std::vector<BlkItem> items;
        const u64 s = 2 * sp;
        const unsigned zrow = (unsigned)((k1 * g.rb2 + s) * g.lc + kc);
        const unsigned zv = (s + 1 < g.rb2 ? 1u : 0u) | (s + 2 < g.rb2 ? 2u : 0u);
        for (u64 j1 = lo1; j1 < hi1; j1++) {
          const u64 m1 = k1 - j1;
          for (u64 ap = 0; ap < nxp && ap <= sp; ap++) {
            const u64 bp = sp - ap;
            if (bp >= nyp) continue;
            for (u64 jc = 0; jc < g.lc; jc++)
              for (u64 mc = 0; mc < g.lc; mc++) {
                unsigned kind;
                if (jc + mc == kc) kind = 0;
                else if (jc + mc + 1 == kc) kind = 1;
                else continue;
                BlkItem it;
                it.xoff = (unsigned)(j1 * g.xplane + (2 * ap * g.lc + jc) * g.row);
                it.yoff = (unsigned)(m1 * g.yplane + (2 * bp * g.lc + mc) * g.row);
                it.zrow = zrow;
                it.kind = kind;
                it.zv = zv;
                items.push_back(it);
              }
          }
        }
        if (!items.empty()) blocks->push_back(std::move(items));
      }
  }
}

static bool blk_dense(const BlkGeom& g) {
  return g.xb1 == g.rb1 && g.yb1 == g.rb1 && g.xb2 == g.rb2 && g.yb2 == g.rb2 && g.rb2 % 4 == 0 &&
         (g.fold_b1 || g.rb1 % 2 == 0);
}

static uint2 blk_entry(const BlkGeom& g, const BlkItem& it, int gi) {
  uint2 e;
  e.x = (it.xoff + (unsigned)(gi * g.xslab)) | ((unsigned)gi << 20) | (it.kind << 24) | (it.zv << 25) | BE_VALID;
  e.y = (it.yoff + (unsigned)(gi * g.yslab)) | (it.zrow << 20);
  return e;
}

// Structured ("folded") table for dense cube slabs: X, Y and Z have the same even plane count D1 (or the slab
// is a single plane) and the same row count D2 = 2P with P even.  A lane is (c1, d[, g]):
//   c1 in 0..D1/2-1 : owns output planes c1 and D1-1-c1  -> D1+1 plane steps (s1 <= c1: plane c1, j1 = s1;
//                                                            s1 > c1: plane D1-1-c1, j1 = s1-c1-1)
//   d  in 0..P/2-1  : owns output row pairs d and P-1-d  -> P+1 pair steps (ap = 0..half, bp = half-ap)
// so every lane executes exactly the same number of items per slab pair, of the same kinds in the same order,
// and touches only 4*Lc output row blocks.  Lanes of a quarter-warp differ only in c1 (3-axis slab) or in the
// staged slab g (single-plane slab): the rows they read at one step are either identical (broadcast) or lie in
// different planes / slabs, whose strides are odd multiples of 16 bytes -> (almost) conflict-free LDS.128.
// T teams share a lane's sequence round-robin (thread = team*lanes + lane).
static bool build_fold_table(const BlkGeom& g, std::vector<uint2>* table, int* n_lo, int* n_hi) {
  if (!blk_dense(g) || g.fold_b1) return false;
  const int D1 = (int)g.rb1, P = (int)(g.rb2 / 2);
  const int C1 = D1 / 2, DD = P / 2;
  const int nl = C1 * DD;
  if (nl > BT || nl < 16) return false;
  const int T = BT / nl;
  std::vector<std::vector<uint2>> seq_lo(nl), seq_hi(nl);
  for (int d = 0; d < DD; d++)
    for (int c1 = 0; c1 < C1; c1++) {
      const int lane = d * C1 + c1;
      int seam = 0;
      for (int phase = 0; phase < 2; phase++) {
        const int half = phase == 0 ? d : P - 1 - d;
        const int s = 2 * half;
        for (int kc = 0; kc < (int)g.lc; kc++)
          for (int gi = 0; gi < g.G; gi++, seam++)
            // D1+1 plane steps in lockstep over the lanes: t <= c1 -> plane c1, j1 = t; t > c1 -> plane D1-1-c1,
            // j1 = t-c1-1 (walked backwards on odd seams so the plane at the seam stays in registers)
            for (int tt = 0; tt <= D1; tt++) {
              const int t = (seam & 1) ? D1 - tt : tt;
              const int r1 = t <= c1 ? c1 : D1 - 1 - c1;
              const int j1 = t <= c1 ? t : t - c1 - 1;
              for (int ap = 0; ap <= half; ap++) {
                const int bp = half - ap;
                for (int jc = 0; jc < (int)g.lc; jc++)
                  for (int mc = 0; mc < (int)g.lc; mc++) {
                    unsigned kind;
                    if (jc + mc == kc) kind = 0;
                    else if (jc + mc + 1 == kc) kind = 1;
                    else continue;
                    BlkItem it;
                    it.xoff = (unsigned)(j1 * g.xplane + (2 * ap * g.lc + jc) * g.row);
                    it.yoff = (unsigned)((r1 - j1) * g.yplane + (2 * bp * g.lc + mc) * g.row);
                    it.zrow = (unsigned)(((u64)r1 * g.rb2 + s) * g.lc + kc);
                    it.kind = kind;
                    it.zv = ((u64)s + 1 < g.rb2 ? 1u : 0u) | ((u64)s + 2 < g.rb2 ? 2u : 0u);
                    (kind ? seq_hi : seq_lo)[lane].push_back(blk_entry(g, it, gi));
                  }
              }
            }
      }
    }
  const size_t len_lo = seq_lo[0].size(), len_hi = seq_hi[0].size();
  for (int l = 0; l < nl; l++)
    if (seq_lo[l].size() != len_lo || seq_hi[l].size() != len_hi) return false;   // not a perfect fold
  *n_lo = (int)((len_lo + T - 1) / T);
  *n_hi = (int)((len_hi + T - 1) / T);
  table->assign((size_t)std::max(*n_lo + *n_hi, 1) * BT, make_uint2(0u, 0u));
  // each team takes a CONTIGUOUS share of the lane's sequence: few output-block changes per thread
  for (int team = 0; team < T; team++)
    for (int l = 0; l < nl; l++) {
      const int tid = team * nl + l;
      size_t b = len_lo * team / T, e = len_lo * (team + 1) / T;
      for (size_t i = b; i < e; i++) (*table)[(i - b) * BT + tid] = seq_lo[l][i];
      b = len_hi * team / T, e = len_hi * (team + 1) / T;
      for (size_t i = b; i < e; i++) (*table)[((size_t)*n_lo + (i - b)) * BT + tid] = seq_hi[l][i];
    }
  return true;
}

struct BlkPlan : DfmaPlan {
  BlkP p;
  BlkGeom g;
};

template <int LT> static void blk_launch_lt(Ctx& ctx, const BlkPlan& pl, const BlkP& p) {
  if (pl.g.lc > 1) {
    allow_dyn_smem(k_mul_blk<LT, true>, ctx.device, pl.g.smem);
    GTP_LAUNCH(ctx, (k_mul_blk<LT, true>), pl.n_units, BT, pl.g.smem, p);
  } else {
    allow_dyn_smem(k_mul_blk<LT, false>, ctx.device, pl.g.smem);
    GTP_LAUNCH(ctx, (k_mul_blk<LT, false>), pl.n_units, BT, pl.g.smem, p);
  }
}

void launch_mul_blk(Ctx& ctx, const MulArgs& a) {
  BlkGeom g;
  GTP_CHECK(blk_geom(a, &g), GTP_ERR_ARG, "blocked product kernel not applicable");
  std::shared_ptr<void>& slot = dfma_plan_slot(ctx.blk_plans, a, 0);
  if (!slot) {
    auto pl = std::make_shared<BlkPlan>();
    pl->g = g;
    BlkP& p = pl->p;
    memset(&p, 0, sizeof(p));
    const int nd = g.nd, na = g.na;
    Shape xst(nd, 1), yst(nd, 1);
    for (int i = nd - 2; i >= 0; --i) {
      xst[i] = xst[i + 1] * a.xs[i + 1];
      yst[i] = yst[i + 1] * a.ys[i + 1];
    }
    p.na = na;
    for (int d = 0; d < na; d++) {
      p.xa[d] = (unsigned)a.xs[d];
      p.ya[d] = (unsigned)a.ys[d];
      p.ra[d] = (unsigned)a.rs[d];
      p.xastr[d] = (long long)xst[d];
      p.yastr[d] = (long long)yst[d];
    }
    p.rows_a0 = (unsigned)a.row_count;
    p.x_planes = (unsigned)g.xb1; p.x_prow = (unsigned)(g.xb2 * g.lc);
    p.y_planes = (unsigned)g.yb1; p.y_prow = (unsigned)(g.yb2 * g.lc);
    p.z_rows = (unsigned)(g.rb1 * g.rb2 * g.lc);
    p.z_pair_stride = (unsigned)g.lc;
    p.x_plane_sm = (unsigned)g.xplane; p.y_plane_sm = (unsigned)g.yplane;
    p.x_slab_sm = (unsigned)g.xslab; p.y_slab_sm = (unsigned)g.yslab;
    p.x_pair_off = p.y_pair_off = (unsigned)(g.lc * g.row);
    p.G = g.G;
    // ---- item table: folded for dense cube slabs, else z-block major, then g, then the block's items, dealt evenly ----
    std::vector<uint2> table;
    int n_lo = 0, n_hi = 0;
    if (!build_fold_table(g, &table, &n_lo, &n_hi)) {
      std::vector<std::vector<BlkItem>> blocks;
      build_items(g, &blocks);
      std::vector<uint2> seq[2];   // by kind
      for (const auto& blk : blocks)
        for (int gi = 0; gi < g.G; gi++)
          for (const BlkItem& it : blk) seq[it.kind].push_back(blk_entry(g, it, gi));
      n_lo = (int)((seq[0].size() + BT - 1) / BT);
      n_hi = (int)((seq[1].size() + BT - 1) / BT);
      table.assign((size_t)std::max(n_lo + n_hi, 1) * BT, make_uint2(0u, 0u));
      for (int kind = 0; kind < 2; kind++) {
        const size_t T = seq[kind].size();
        const size_t base = kind ? (size_t)n_lo : 0;
        for (int t = 0; t < BT; t++) {
          size_t b = T * t / BT, e = T * (t + 1) / BT;
          for (size_t i = b; i < e; i++) table[(base + (i - b)) * BT + t] = seq[kind][i];
        }
      }
    }
    p.nsteps_lo = n_lo;
    p.nsteps = n_lo + n_hi;
    const Shape axs(a.xs.begin(), a.xs.begin() + na), ays(a.ys.begin(), a.ys.begin() + na), ars(a.rs.begin(), a.rs.begin() + na);
    dfma_upload(ctx, pl.get(), table, dfma_units(a, axs, ays, ars, g.G, (u64)ctx.sm_count * 2));
    p.table = reinterpret_cast<const uint2*>(pl->table->d);
    p.units = reinterpret_cast<const uint4*>(pl->units->d);
    slot = pl;
  }
  const BlkPlan& pl = *std::static_pointer_cast<BlkPlan>(slot);
  BlkP p = pl.p;
  p.x = a.x;
  p.y = a.y;
  p.out = a.out;
  u64 row_elems = 1;
  for (int d = 1; d < a.ndim; d++) row_elems *= a.rs[d];
  GTP_CUDA(cudaMemsetAsync(a.out, 0, a.row_count * row_elems * sizeof(double), ctx.stream));
  if (pl.n_units == 0 || p.nsteps == 0) return;
  switch ((int)pl.g.lt) {
    case 8: blk_launch_lt<8>(ctx, pl, p); break;
    case 10: blk_launch_lt<10>(ctx, pl, p); break;
    case 12: blk_launch_lt<12>(ctx, pl, p); break;
    case 14: blk_launch_lt<14>(ctx, pl, p); break;
    case 16: blk_launch_lt<16>(ctx, pl, p); break;
    default: throw Error(GTP_ERR_ARG, "unsupported chunk length");
  }
}

}  // namespace gtp
