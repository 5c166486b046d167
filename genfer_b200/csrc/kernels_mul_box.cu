// DFMA product for tensors with more than 8 effective axes (plan kind 8).
//
// Evaluation tensors have one axis per live program variable, most of them short (extents 2-7): the sliding and blocked
// kernels need a last axis of at least 8 and at most 6 leading axes, and the reference-order kernel runs such products at
// 0.02-0.09 TFLOP/s (one thread per output, a 1-4 term innermost sum, an odometer over up to 23 axes per step).  Here the
// axes are split into leading axes and a trailing box of the last few axes (at most 256 result coefficients):
//   * a work unit is (output leading index, chunk of the leading J box), built and LPT-sorted by dfma_units;
//   * the CTA runs G groups of threads, each stages one (J, K - J) pair of X and Y boxes per round with cp.async
//     (16-byte copies when the boxes have an even length and the operands are 16-byte aligned, else 8-byte ones);
//   * a host-built pair table of the trailing box (every (x, y) coefficient pair of every box output, packed 16 + 16 bit)
//     sits in shared memory; it is cut into segments of at most P / gt pairs, and each thread owns up to R segments
//     (LPT-dealt), accumulated in registers with DFMA over the whole chunk;
//   * partial outputs of a unit (a segment per thread, a chunk per unit) meet in HBM through RED.ADD.F64.
// Summation order differs from the reference's: tolerance-checked like the other DFMA kernels (exact on small integers).
#include <algorithm>

#include "kernels.cuh"

namespace gtp {

namespace {

constexpr int BX_BT = 128;          // threads per CTA
constexpr int BX_R = 8;             // pair-table segments (register accumulators) per thread
constexpr u64 BX_MAX_ZBOX = 256;    // result coefficients of the trailing box
constexpr u64 BX_MAX_PAIRS = 8192;  // pairs of the trailing box (32 KB of shared memory)
constexpr u64 BX_MAX_SMEM = 96 * 1024;

struct BoxP {
  int na;                            // leading axes (axis 0: the row axis)
  unsigned rows_a0;
  unsigned xa[MAXD], ya[MAXD], ra[MAXD];
  long long xastr[MAXD], yastr[MAXD];
  unsigned xbox, ybox, zbox;         // coefficients of the trailing boxes (contiguous in X, Y, Z)
  unsigned xbox_sm, ybox_sm;         // their staging lengths (rounded up to even)
  unsigned G, gt;                    // groups per CTA, threads per group
  unsigned npairs;
  int v16;                           // 16-byte copies
  const uint4* slots;                // [gt * BX_R]: (box output, pair begin, pair end, -)
  const unsigned* pairs;             // x index | y index << 16, grouped by box output
  const uint4* units;
  const double* x;
  const double* y;
  double* out;
};

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}

__global__ void __launch_bounds__(BX_BT) k_mul_box(const __grid_constant__ BoxP p) {
  extern __shared__ __align__(16) double smem[];
  __shared__ unsigned s_k[MAXD], s_lo[MAXD], s_ext[MAXD];
  double* Xs = smem;
  double* Ys = smem + (size_t)p.G * p.xbox_sm;
  unsigned* pairs = reinterpret_cast<unsigned*>(Ys + (size_t)p.G * p.ybox_sm);
  const unsigned tid = threadIdx.x, g = tid / p.gt, lt = tid - g * p.gt;
  const uint4 unit = p.units[blockIdx.x];

  for (unsigned i = tid; i < p.npairs; i += BX_BT) pairs[i] = p.pairs[i];
  if (tid == 0) {   // the unit's output leading index and its J box
    unsigned rem = unit.x;
    for (int a = p.na - 1; a >= 0; --a) {
      const unsigned len = (a == 0) ? p.rows_a0 : p.ra[a];
      const unsigned idx = rem % len;
      rem /= len;
      const unsigned k = (a == 0) ? unit.w : idx;
      const unsigned l = (k + 1 > p.ya[a]) ? k + 1 - p.ya[a] : 0;
      const unsigned h = (k + 1 < p.xa[a]) ? k + 1 : p.xa[a];
      s_k[a] = k;
      s_lo[a] = l;
      s_ext[a] = h > l ? h - l : 0;
    }
  }
  unsigned sz[BX_R], sb[BX_R], se[BX_R];
#pragma unroll
  for (int r = 0; r < BX_R; r++) {
    const uint4 s = p.slots[lt * BX_R + r];
    sz[r] = s.x;
    sb[r] = s.y;
    se[r] = s.z;
  }
  double acc[BX_R];
#pragma unroll
  for (int r = 0; r < BX_R; r++) acc[r] = 0.0;
  const double* xs = Xs + (size_t)g * p.xbox_sm;
  const double* ys = Ys + (size_t)g * p.ybox_sm;

  for (unsigned q = unit.y; q < unit.z; q += p.G) {
    __syncthreads();   // the previous round's boxes are consumed (first round: the J box and the pair table are written)
    const unsigned jq = q + g;
    const bool active = g < p.G && jq < unit.z;
    if (active) {
      long long xo = 0, yo = 0;
      unsigned rem = jq;
      for (int a = p.na - 1; a >= 0; --a) {
        const unsigned e = s_ext[a];
        const unsigned j = s_lo[a] + rem % e;
        rem /= e;
        xo += (long long)j * p.xastr[a];
        yo += (long long)(s_k[a] - j) * p.yastr[a];
      }
      double* dx = Xs + (size_t)g * p.xbox_sm;
      double* dy = Ys + (size_t)g * p.ybox_sm;
      if (p.v16) {
        for (unsigned i = lt; 2 * i < p.xbox; i += p.gt) cp_async16(dx + 2 * i, p.x + xo + 2 * i);
        for (unsigned i = lt; 2 * i < p.ybox; i += p.gt) cp_async16(dy + 2 * i, p.y + yo + 2 * i);
      } else {
        for (unsigned i = lt; i < p.xbox; i += p.gt) cp_async8(dx + i, p.x + xo + i);
        for (unsigned i = lt; i < p.ybox; i += p.gt) cp_async8(dy + i, p.y + yo + i);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    if (active) {
#pragma unroll
      for (int r = 0; r < BX_R; r++) {
        double s = acc[r];
        for (unsigned i = sb[r]; i < se[r]; i++) {
          const unsigned e = pairs[i];
          s = fma(xs[e & 0xffffu], ys[e >> 16], s);
        }
        acc[r] = s;
      }
    }
  }
  if (g < p.G) {
    double* dst = p.out + (size_t)unit.x * p.zbox;
#pragma unroll
    for (int r = 0; r < BX_R; r++)
      if (se[r] > sb[r]) atomicAdd(dst + sz[r], acc[r]);   // RED.ADD.F64: the result is unused
  }
}

struct BoxGeom {
  int na = 0;
  u64 xbox = 0, ybox = 0, zbox = 0, npairs = 0;
  unsigned gt = 0, G = 0;
  size_t smem = 0;
};

unsigned box_gt(u64 zbox) {   // threads per group: gt * (R - 1) >= zbox leaves room for the split segments
  unsigned gt = 32;
  while ((u64)gt * (BX_R - 1) < zbox) gt *= 2;
  return gt;
}

// The widest trailing box within the limits; false: no box, or the product is not this kernel's.
bool box_geom(const MulArgs& a, BoxGeom* g) {
  const int nd = a.ndim;
  if (nd < 2 || nd > MAXD || a.accumulate) return false;
  int ne = 0;
  for (int d = 0; d < nd; d++) ne += a.rs[d] != 1;
  if (ne <= 8) return false;
  for (int nb = 1; nb < nd; nb++) {
    const Shape txs(a.xs.end() - nb, a.xs.end()), tys(a.ys.end() - nb, a.ys.end()), trs(a.rs.end() - nb, a.rs.end());
    const u64 xb = prod(txs), yb = prod(tys), zb = prod(trs);
    const double pairs = mul_macs(txs, tys, trs);
    if (zb > BX_MAX_ZBOX || pairs > (double)BX_MAX_PAIRS || xb >= 65536 || yb >= 65536) break;
    const unsigned gt = box_gt(zb);
    const unsigned G = BX_BT / gt;
    const size_t smem = (size_t)G * ((xb + 1) / 2 * 2 + (yb + 1) / 2 * 2) * sizeof(double) + (size_t)pairs * sizeof(unsigned);
    if (smem > BX_MAX_SMEM) break;
    g->na = nd - nb;
    g->xbox = xb; g->ybox = yb; g->zbox = zb; g->npairs = (u64)pairs;
    g->gt = gt; g->G = G; g->smem = smem;
  }
  if (g->na == 0 || g->npairs == 0) return false;
  // 32-bit unit fields: output leading indices and J-box positions
  const u64 rows = a.rows.empty() ? a.row_count : a.rows.size();
  u64 slabs = rows, jbox = 1;
  for (int d = 0; d < g->na; d++) {
    if (d) slabs *= a.rs[d];
    jbox *= std::min(a.xs[d], a.ys[d]);
  }
  return slabs < (1ull << 32) && jbox < (1ull << 31);
}

// Pair table of the trailing box: per box output (row-major), its (x, y) pairs; cut into segments of at most P / gt pairs
// and dealt longest first to the least-loaded thread with a free slot.
void box_table(const MulArgs& a, const BoxGeom& g, std::vector<uint4>* slots, std::vector<unsigned>* pairs) {
  const int nd = a.ndim, nb = nd - g.na;
  const Shape txs(a.xs.end() - nb, a.xs.end()), tys(a.ys.end() - nb, a.ys.end()), trs(a.rs.end() - nb, a.rs.end());
  Shape xst(nb, 1), yst(nb, 1);
  for (int i = nb - 2; i >= 0; --i) {
    xst[i] = xst[i + 1] * txs[i + 1];
    yst[i] = yst[i + 1] * tys[i + 1];
  }
  struct Seg { unsigned z, b, e; };
  std::vector<Seg> segs;
  const u64 cap = std::max<u64>(1, (g.npairs + g.gt - 1) / g.gt);
  std::vector<u64> k(nb), lo(nb), hi(nb), j(nb);
  for (u64 z = 0; z < g.zbox; z++) {
    u64 rem = z;
    bool empty = false;
    for (int d = nb - 1; d >= 0; --d) {
      k[d] = rem % trs[d];
      rem /= trs[d];
      lo[d] = sat_sub(k[d] + 1, tys[d]);
      hi[d] = std::min<u64>(k[d] + 1, txs[d]);
      empty |= hi[d] <= lo[d];
      j[d] = lo[d];
    }
    if (empty) continue;
    const unsigned begin = (unsigned)pairs->size();
    while (true) {
      u64 xi = 0, yi = 0;
      for (int d = 0; d < nb; d++) {
        xi += j[d] * xst[d];
        yi += (k[d] - j[d]) * yst[d];
      }
      pairs->push_back((unsigned)xi | (unsigned)yi << 16);
      int d = nb - 1;
      for (; d >= 0; --d) {
        if (++j[d] < hi[d]) break;
        j[d] = lo[d];
      }
      if (d < 0) break;
    }
    for (unsigned b = begin; b < pairs->size(); b += (unsigned)cap)
      segs.push_back({(unsigned)z, b, (unsigned)std::min<u64>(pairs->size(), b + cap)});
  }
  std::stable_sort(segs.begin(), segs.end(), [](const Seg& x, const Seg& y) { return x.e - x.b > y.e - y.b; });
  std::vector<u64> load(g.gt, 0);
  std::vector<int> used(g.gt, 0);
  slots->assign((size_t)g.gt * BX_R, make_uint4(0u, 0u, 0u, 0u));
  for (const Seg& s : segs) {
    int best = -1;
    for (unsigned t = 0; t < g.gt; t++)
      if (used[t] < BX_R && (best < 0 || load[t] < load[best])) best = (int)t;
    GTP_CHECK(best >= 0, GTP_ERR_ARG, "box product: pair table does not fit the thread slots");
    (*slots)[(size_t)best * BX_R + used[best]++] = make_uint4(s.z, s.b, s.e, 0u);
    load[best] += s.e - s.b;
  }
}

struct BoxPlan : DfmaPlan {
  BoxP p;
  BoxGeom g;
};

}  // namespace

bool box_mul_applicable(const Ctx& ctx, const MulArgs& a) {
  BoxGeom g;
  return box_geom(a, &g);
}

void launch_mul_box(Ctx& ctx, const MulArgs& a) {
  BoxGeom g;
  GTP_CHECK(box_geom(a, &g), GTP_ERR_ARG, "box product kernel not applicable");
  std::shared_ptr<void>& slot = dfma_plan_slot(ctx.box_plans, a, 0);
  if (!slot) {
    auto pl = std::make_shared<BoxPlan>();
    pl->g = g;
    BoxP& p = pl->p;
    memset(&p, 0, sizeof(p));
    const int nd = a.ndim, na = g.na;
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
    p.xbox = (unsigned)g.xbox; p.ybox = (unsigned)g.ybox; p.zbox = (unsigned)g.zbox;
    p.xbox_sm = (unsigned)((g.xbox + 1) / 2 * 2); p.ybox_sm = (unsigned)((g.ybox + 1) / 2 * 2);
    p.G = g.G; p.gt = g.gt;
    p.npairs = (unsigned)g.npairs;
    std::vector<uint4> slots;
    std::vector<unsigned> pairs;
    box_table(a, g, &slots, &pairs);
    // one device table: the slots (two uint2 each), then the pairs (two per uint2)
    std::vector<uint2> table;
    for (const uint4& s : slots) {
      table.push_back(make_uint2(s.x, s.y));
      table.push_back(make_uint2(s.z, s.w));
    }
    for (size_t i = 0; i < pairs.size(); i += 2) table.push_back(make_uint2(pairs[i], i + 1 < pairs.size() ? pairs[i + 1] : 0u));
    const Shape axs(a.xs.begin(), a.xs.begin() + na), ays(a.ys.begin(), a.ys.begin() + na), ars(a.rs.begin(), a.rs.begin() + na);
    dfma_upload(ctx, pl.get(), table, dfma_units(a, axs, ays, ars, (int)g.G, (u64)ctx.sm_count * 4));
    p.slots = reinterpret_cast<const uint4*>(pl->table->d);
    p.pairs = reinterpret_cast<const unsigned*>(pl->table->d + slots.size() * 2);
    p.units = reinterpret_cast<const uint4*>(pl->units->d);
    slot = pl;
  }
  const BoxPlan& pl = *std::static_pointer_cast<BoxPlan>(slot);
  BoxP p = pl.p;
  p.x = a.x;
  p.y = a.y;
  p.out = a.out;
  p.v16 = pl.g.xbox % 2 == 0 && pl.g.ybox % 2 == 0 && !((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.y)) & 15u);
  u64 row_elems = 1;
  for (int d = 1; d < a.ndim; d++) row_elems *= a.rs[d];
  GTP_CUDA(cudaMemsetAsync(a.out, 0, a.row_count * row_elems * sizeof(double), ctx.stream));
  if (pl.n_units == 0) return;
  allow_dyn_smem(k_mul_box, ctx.device, pl.g.smem);
  GTP_LAUNCH(ctx, k_mul_box, pl.n_units, BX_BT, pl.g.smem, p);
}

}  // namespace gtp
