// Truncated N-D Taylor product (multivariate_taylor.rs:972-1012) -- reference-order kernel,
// kernel selection, MAC counting and the FP64 pipe probes.
//
// k_mul_ordered is the general kernel: any shapes, any row subset, one thread per output
// coefficient.  It performs the multiply and the add separately (DMUL + DADD, no FMA) and
// in exactly the reference's nesting order -- outer axes ascending, the innermost non-unit axis
// summed from zero and then added (mul_1d :972-982 feeding `*z += o` :998) -- so its results are
// bit-identical to the reference f64 path.  The DFMA kernels live in kernels_mul_blk.cu and kernels_mul_slide.cu
// (their shared host plan path is here); launch_mul() picks between them.
#include <algorithm>

#include "kernels.cuh"

namespace gtp {

constexpr int MUL_MAXE = 8;  // effective (non-unit) result axes handled with register odometers

struct MulP {
  int ne;                       // effective axes
  int row_axis;                 // 1 if effective axis 0 is the (sharded) leading axis
  unsigned xs[MAXD], ys[MAXD], rs[MAXD];
  long long xstr[MAXD], ystr[MAXD];
  u64 row_begin, row_step, row_count;
  u64 row_elems;                // prod of rs over the non-row effective axes
  u64 total;                    // outputs computed by this launch
  const double* x;
  const double* y;
  double* out;
  int accumulate;
};

template <int NE> __device__ __forceinline__ void mul_ordered_body(const MulP& p);
template <int NE>
__global__ void __launch_bounds__(128) k_mul_ordered(const MulP p) { mul_ordered_body<NE>(p); }
// Single-CTA variant for small results (<= 1024 coefficients): the producer classifies its own output (extract_linear scan,
// kernels.cuh::cls_epilogue) instead of a separate classification launch + wait by the next operator's dispatch.
template <int NE>
__global__ void __launch_bounds__(1024) k_mul_ordered_cls(const MulP p, const FusedClsArgs cls) {
  mul_ordered_body<NE>(p);
  if (cls.slot) cls_epilogue(p.out, cls.p, cls.slot, cls.seq);
}
template <int NE>
__device__ __forceinline__ void mul_ordered_body(const MulP& p) {
  const u64 gstride = (u64)gridDim.x * blockDim.x;
  for (u64 lin = (u64)blockIdx.x * blockDim.x + threadIdx.x; lin < p.total; lin += gstride) {
    unsigned k[NE], lo[NE], hi[NE];
    u64 rem = lin;
    bool empty = false;
#pragma unroll
    for (int d = NE - 1; d >= 0; --d) {
      if (d == 0 && p.row_axis) {
        k[d] = (unsigned)(p.row_begin + rem * p.row_step);
      } else {
        k[d] = (unsigned)(rem % p.rs[d]);
        rem /= p.rs[d];
      }
      unsigned l = (k[d] + 1 > p.ys[d]) ? k[d] + 1 - p.ys[d] : 0;   // :975 / :1002
      unsigned h = (k[d] + 1 < p.xs[d]) ? k[d] + 1 : p.xs[d];       // :976 / :1003
      lo[d] = l;
      hi[d] = h;
      empty |= (h <= l);
    }
    double total = p.accumulate ? p.out[lin] : 0.0;
    if (!empty) {
      unsigned j[NE];
      long long xo = 0, yo = 0;
#pragma unroll
      for (int d = 0; d < NE - 1; d++) {
        j[d] = lo[d];
        xo += (long long)lo[d] * p.xstr[d];
        yo += (long long)(k[d] - lo[d]) * p.ystr[d];
      }
      const long long xsl = p.xstr[NE - 1], ysl = p.ystr[NE - 1];
      const unsigned kl = k[NE - 1], lol = lo[NE - 1], hil = hi[NE - 1];
      while (true) {
        // innermost non-unit axis: summed from zero, then added (mul_1d + `*z += o`)
        double inner = 0.0;
        const double* xp = p.x + xo + (long long)lol * xsl;
        const double* yp = p.y + yo + (long long)(kl - lol) * ysl;
        for (unsigned jl = lol; jl < hil; jl++) {
          inner = __dadd_rn(inner, __dmul_rn(*xp, *yp));
          xp += xsl;
          yp -= ysl;
        }
        total = __dadd_rn(total, inner);
        // odometer over the outer effective axes, last one fastest (the recursion order)
        bool advanced = false;
#pragma unroll
        for (int dd = NE - 2; dd >= 0; --dd) {
          if (!advanced) {
            if (++j[dd] < hi[dd]) {
              xo += p.xstr[dd];
              yo -= p.ystr[dd];
              advanced = true;
            } else {
              xo -= (long long)(hi[dd] - 1 - lo[dd]) * p.xstr[dd];
              yo += (long long)(hi[dd] - 1 - lo[dd]) * p.ystr[dd];
              j[dd] = lo[dd];
            }
          }
        }
        if (!advanced) break;  // wrapped around every axis (or NE == 1)
      }
    }
    p.out[lin] = total;
  }
}

// MACs of the rows a launch computes (the `lo..hi` trip counts of :975-977, :1002-1004)
double args_macs(const MulArgs& a) {
  double total = 1.0;
  for (int d = 0; d < a.ndim; d++) {
    double s = 0;
    auto trips = [&](u64 k) {
      u64 lo = sat_sub(k + 1, a.ys[d]), hi = std::min<u64>(k + 1, a.xs[d]);
      return hi > lo ? (double)(hi - lo) : 0.0;
    };
    if (d == 0) {
      if (!a.rows.empty()) for (u64 k : a.rows) s += trips(k);
      else for (u64 i = 0; i < a.row_count; i++) s += trips(a.row_begin + i * a.row_step);
    } else {
      for (u64 k = 0; k < a.rs[d]; k++) s += trips(k);
    }
    total *= s;
  }
  return total;
}

double mul_macs(const Shape& xs, const Shape& ys, const Shape& rs) {
  double total = 1.0;
  for (size_t a = 0; a < rs.size(); a++) {
    double s = 0;
    for (u64 k = 0; k < rs[a]; k++) {
      u64 lo = sat_sub(k + 1, ys[a]), hi = std::min<u64>(k + 1, xs[a]);
      if (hi > lo) s += (double)(hi - lo);
    }
    total *= s;
  }
  return total;
}

// ------------------------------------------------------------------------------------------
// Host plan path shared by the DFMA kernels (kernels_mul_blk.cu, kernels_mul_slide.cu)
// ------------------------------------------------------------------------------------------
u64 dfma_chunk(u64 l) {
  for (u64 lt : {16, 14, 12, 10, 8})
    if (l % lt == 0) return lt;
  return 0;
}

std::vector<uint4> dfma_units(const MulArgs& a, const Shape& axs, const Shape& ays, const Shape& ars, int G, u64 slots) {
  const int na = (int)axs.size();
  u64 n_slabs = a.row_count;
  for (int d = 1; d < na; d++) n_slabs *= ars[d];
  auto row_of = [&](u64 idx) -> u64 { return a.rows.empty() ? a.row_begin + idx * a.row_step : a.rows[idx]; };
  std::vector<u64> boxes(n_slabs);
  std::vector<unsigned> k0s(n_slabs, 0);
  u64 total_pairs = 0;
  for (u64 s = 0; s < n_slabs; s++) {
    u64 rem = s, box = 1;
    for (int d = na - 1; d >= 0; --d) {
      u64 len = (d == 0) ? a.row_count : ars[d];
      u64 idx = rem % len;
      rem /= len;
      u64 k = (d == 0) ? row_of(idx) : idx;
      if (d == 0) k0s[s] = (unsigned)k;
      u64 lo = sat_sub(k + 1, ays[d]), hi = std::min(k + 1, axs[d]);
      box *= hi > lo ? hi - lo : 0;
    }
    boxes[s] = box;
    total_pairs += box;
  }
  // at least 8 rounds per unit amortise its set-up -- unless that leaves resident-CTA slots empty (mid-size products)
  const u64 min_chunk = total_pairs >= slots * 8 * (u64)G ? 8 * (u64)G : (u64)G;
  u64 chunk = std::max<u64>(min_chunk, total_pairs / (slots * 16) + 1);
  chunk = (chunk + G - 1) / G * G;   // whole rounds
  std::vector<uint4> units;
  for (u64 s = 0; s < n_slabs; s++) {
    u64 box = boxes[s];
    if (!box) continue;
    u64 parts = (box + chunk - 1) / chunk;
    u64 per = (box + parts - 1) / parts;
    per = (per + G - 1) / G * G;
    for (u64 q0 = 0; q0 < box; q0 += per) units.push_back(make_uint4((unsigned)s, (unsigned)q0, (unsigned)std::min(box, q0 + per), k0s[s]));
  }
  std::stable_sort(units.begin(), units.end(), [](const uint4& x, const uint4& y) { return (x.z - x.y) > (y.z - y.y); });
  return units;
}

using DfmaPlanCache = std::map<std::vector<u64>, std::shared_ptr<void>>;
std::shared_ptr<void>& dfma_plan_slot(std::shared_ptr<void>& cache, const MulArgs& a, u64 extra) {
  if (!cache) cache = std::make_shared<DfmaPlanCache>();
  auto& plans = *std::static_pointer_cast<DfmaPlanCache>(cache);
  std::vector<u64> key{(u64)a.ndim};   // fixes where the shapes end and the row list begins
  key.insert(key.end(), a.xs.begin(), a.xs.end());
  key.insert(key.end(), a.ys.begin(), a.ys.end());
  key.insert(key.end(), a.rs.begin(), a.rs.end());
  key.push_back(a.row_begin);
  key.push_back(a.row_step);
  key.push_back(a.row_count);
  key.push_back(extra);
  key.insert(key.end(), a.rows.begin(), a.rows.end());
  auto it = plans.find(key);
  if (it != plans.end()) return it->second;
  if (plans.size() > 64) plans.clear();
  return plans[key];
}

void dfma_upload(Ctx& ctx, DfmaPlan* pl, const std::vector<uint2>& table, const std::vector<uint4>& units) {
  pl->n_units = (unsigned)units.size();
  pl->table = ctx.alloc(table.size() + 1);   // sizes in doubles: a uint2 is one, a uint4 two
  pl->units = ctx.alloc(units.size() * 2 + 1);
  if (!table.empty())
    GTP_CUDA(cudaMemcpyAsync(pl->table->d, table.data(), table.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx.stream));
  if (!units.empty())
    GTP_CUDA(cudaMemcpyAsync(pl->units->d, units.data(), units.size() * sizeof(uint4), cudaMemcpyHostToDevice, ctx.stream));
  ctx.sync();   // the host arrays are the caller's temporaries
}

// implemented in kernels_mul_blk.cu / kernels_mul_slide.cu
bool blk_mul_applicable(const Ctx& ctx, const MulArgs& a);
void launch_mul_blk(Ctx& ctx, const MulArgs& a);
bool slide_mul_applicable(const Ctx& ctx, const MulArgs& a);
void launch_mul_slide(Ctx& ctx, const MulArgs& a);
bool launch_mul_axis(Ctx& ctx, const MulArgs& a);   // kernels_mul_axis.cu
bool launch_stencil_rows(Ctx& ctx, const MulArgs& a);   // kernels_horner.cu: row-staged (bulk-copy) small-operand product

// 0: reference-order kernel, 2: 2x2-blocked DFMA kernel (kernels_mul_blk.cu), 3: sliding 1x2 DFMA kernel for dense
// cube slabs (kernels_mul_slide.cu).  (1 was the cube-16-only kernel of
// the first round; the blocked kernel with folded tables superseded it.)
static int pad_plan(const Ctx& ctx, const MulArgs& a, MulArgs* out_best);
// what launch_mul() will run -- 0: reference-order family (reference-order kernel, small-operand stencil, axis convolution:
// all bit-exact), 2 / 3: blocked / sliding DFMA kernel, 6 / 7: the same after zero-extending odd extents
int mul_plan_kind(const Ctx& ctx, const MulArgs& a) {
  const int k = mul_kernel_kind(ctx, a);
  if (k || !ctx.fast_mul) return k;
  if (ctx.use_stencil && std::min(prod(a.xs), prod(a.ys)) <= (u64)32 && std::max(prod(a.xs), prod(a.ys)) >= 4096) return 0;
  int nonunit_x = 0, nonunit_y = 0;
  for (int d = 0; d < a.ndim; d++) { nonunit_x += a.xs[d] > 1; nonunit_y += a.ys[d] > 1; }
  if (ctx.use_axis && (nonunit_x == 1) != (nonunit_y == 1)) return 0;   // axis convolution (bit-exact)
  MulArgs best;
  const int pk = pad_plan(ctx, a, &best);
  return pk ? pk + 4 : 0;
}
int mul_kernel_kind(const Ctx& ctx, const MulArgs& a) {
  if (!ctx.fast_mul) return 0;
  if ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.y)) & 15u) return 0;  // cp.async 16-byte staging
  if (ctx.use_stencil && std::min(prod(a.xs), prod(a.ys)) <= (u64)32 && std::max(prod(a.xs), prod(a.ys)) >= 4096) return 0;  // stencil kernel
  if (ctx.use_slide && slide_mul_applicable(ctx, a)) return 3;
  return blk_mul_applicable(ctx, a) ? 2 : 0;
}

static void launch_mul_ordered(Ctx& ctx, const MulArgs& a) {
  const int nd = a.ndim;
  GTP_CHECK(nd <= MAXD, GTP_ERR_ARG, "ndim exceeds GTP_MAX_NDIM");
  MulP p;
  memset(&p, 0, sizeof(p));
  Shape xst(nd, 1), yst(nd, 1);
  for (int i = nd - 2; i >= 0; --i) {
    xst[i] = xst[i + 1] * a.xs[i + 1];
    yst[i] = yst[i + 1] * a.ys[i + 1];
  }
  u64 row_elems = 1;
  for (int i = 1; i < nd; i++) row_elems *= a.rs[i];
  int ne = 0;
  p.row_axis = 0;
  for (int d = 0; d < nd; d++) {
    bool is_row = (d == 0);
    if (a.rs[d] == 1) {
      if (is_row) GTP_CHECK(a.row_count <= 1 && a.row_begin == 0, GTP_ERR_ARG, "row range on a unit leading axis");
      continue;  // unit result axis: only index 0 of both operands contributes
    }
    GTP_CHECK(ne < MUL_MAXE, GTP_ERR_ARG, "more than 8 non-unit result axes are not supported yet");
    if (is_row) p.row_axis = 1;
    p.xs[ne] = (unsigned)a.xs[d];
    p.ys[ne] = (unsigned)a.ys[d];
    p.rs[ne] = (unsigned)a.rs[d];
    p.xstr[ne] = (long long)xst[d];
    p.ystr[ne] = (long long)yst[d];
    ne++;
  }
  if (ne == 0) {  // single coefficient: leaf `*res += x*y` (:988-991)
    p.xs[0] = p.ys[0] = p.rs[0] = 1;
    p.xstr[0] = p.ystr[0] = 1;
    ne = 1;
  }
  p.ne = ne;
  p.row_begin = a.row_begin;
  p.row_step = a.row_step;
  p.row_count = (nd == 0 || a.rs[0] == 1) ? 1 : a.row_count;
  p.row_elems = (nd == 0) ? 1 : row_elems;
  p.total = p.row_count * p.row_elems;
  p.x = a.x;
  p.y = a.y;
  p.out = a.out;
  p.accumulate = a.accumulate ? 1 : 0;
  if (p.total == 0) return;
  // small whole results: one CTA that also classifies what it wrote
  if (p.total <= 1024 && !a.accumulate && a.row_begin == 0 && a.row_step == 1 && (nd == 0 || a.rs[0] == 1 || a.row_count == a.rs[0])) {
    FusedClsArgs cls;
    if (fused_cls_begin(ctx, a.out, a.rs, &cls)) {
      const int blk = (int)std::min<u64>(1024, (p.total + 31) / 32 * 32);
      switch (ne) {
#define CASE(N) case N: GTP_LAUNCH(ctx, k_mul_ordered_cls<N>, 1, blk, 0, p, cls); break;
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
#undef CASE
      }
      return;
    }
  }
  int block = 128;
  int grid = (int)std::max<u64>(1, std::min<u64>((p.total + block - 1) / block, (u64)ctx.sm_count * 64));
  switch (ne) {
#define CASE(N) case N: GTP_LAUNCH(ctx, k_mul_ordered<N>, grid, block, 0, p); break;
    CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
#undef CASE
  }
}

// ------------------------------------------------------------------------------------------
// Stencil product: one operand has at most ST_MAXT coefficients (the multilinear substitutions and thinning
// factors of real programs: X of shape [297, 282, 297] times Y of shape [2, 1, 2] is the typical heavy product of the
// population models).  Such a product is HBM-bound -- a few MACs per output -- and the generic reference-order kernel
// (64-bit odometers, one dependent gather per MAC) reaches ~0.4 TB/s on it.  Here the small operand's coefficients and
// their offsets sit in the kernel parameters / registers; a thread computes one output coefficient with 32-bit index
// arithmetic, its few loads independent of each other.  The terms are visited in the reference's order (outer axes
// ascending in the X index; the innermost non-unit axis summed from zero and then added, :996-998), multiply and add
// separate: bit-identical to the reference-order kernel.
// ------------------------------------------------------------------------------------------
constexpr int ST_MAXT = 32;
struct StencilP {
  int ne, nt, row_axis;
  unsigned rs[MUL_MAXE], big[MUL_MAXE];     // result extents, extents of the big operand (effective axes)
  long long bstr[MUL_MAXE];                 // strides of the big operand
  unsigned char m[ST_MAXT][MUL_MAXE];       // term t pairs small[m_t] with big[k - m_t]
  unsigned char group_start[ST_MAXT];       // 1: first term of a new outer-axes group
  unsigned short sidx[ST_MAXT];             // linear index of m_t in the small operand
  long long delta[ST_MAXT];                 // sum_a m_t[a] * bstr[a]
  unsigned row_begin, row_step;
  unsigned total;                           // coefficients (k_mul_stencil) or units of four (k_mul_stencil_v4)
  unsigned lastq;                           // v4: units per row of the innermost effective axis
  const double* bigp;
  const double* smallp;
  double* out;
};
// NT: compile-time bound on the number of terms (2, 4, 8, 16, 32): with a single 32-term body ptxas predicates all 32
// term bodies and a 4-term product executes ~700 instructions per coefficient.
template <int NE, int NT>
__global__ void __launch_bounds__(256) k_mul_stencil(const __grid_constant__ StencilP p) {
  double sv[NT];
#pragma unroll
  for (int t = 0; t < NT; t++) sv[t] = t < p.nt ? p.smallp[p.sidx[t]] : 0.0;
  const unsigned gstride = gridDim.x * blockDim.x;
  for (unsigned lin = blockIdx.x * blockDim.x + threadIdx.x; lin < p.total; lin += gstride) {
    unsigned k[NE];
    unsigned rem = lin;
    long long base = 0;
#pragma unroll
    for (int d = NE - 1; d >= 0; --d) {
      if (d == 0 && p.row_axis) {
        k[d] = p.row_begin + rem * p.row_step;
      } else {
        const unsigned q = rem / p.rs[d];
        k[d] = rem - q * p.rs[d];
        rem = q;
      }
      base += (long long)k[d] * p.bstr[d];
    }
    double total = 0.0, inner = 0.0;
    bool open = false;    // a group with valid outer axes is being summed
#pragma unroll
    for (int t = 0; t < NT; t++) {
      if (t < p.nt) {
        if (p.group_start[t]) {
          if (open) total = __dadd_rn(total, inner);
          inner = 0.0;
          open = true;
#pragma unroll
          for (int d = 0; d < NE - 1; d++) {
            const unsigned md = p.m[t][d];
            open = open && k[d] >= md && k[d] - md < p.big[d];
          }
        }
        const unsigned ml = p.m[t][NE - 1];
        if (open && k[NE - 1] >= ml && k[NE - 1] - ml < p.big[NE - 1])
          inner = __dadd_rn(inner, __dmul_rn(p.bigp[base - p.delta[t]], sv[t]));
      }
    }
    if (open) total = __dadd_rn(total, inner);
    p.out[lin] = total;
  }
}

// Four consecutive coefficients of the innermost effective axis per thread: the index decode, the outer-axis validity
// tests and the group bookkeeping are shared by the four, which halves the instructions per coefficient again.  The
// per-coefficient order of operations is unchanged.  (The big operand's innermost effective stride is 1: unit result axes
// have unit operands, see launch_mul_stencil.)  p.total counts units of four; p.lastq = ceil(rs_last / 4).
template <int NE, int NT>
__global__ void __launch_bounds__(256) k_mul_stencil_v4(const __grid_constant__ StencilP p) {
  static_assert(NE >= 2, "the innermost effective axis must not be the row axis");
  double sv[NT];
#pragma unroll
  for (int t = 0; t < NT; t++) sv[t] = t < p.nt ? p.smallp[p.sidx[t]] : 0.0;
  const unsigned gstride = gridDim.x * blockDim.x;
  const unsigned rl = p.rs[NE - 1], bl = p.big[NE - 1];
  for (unsigned unit = blockIdx.x * blockDim.x + threadIdx.x; unit < p.total; unit += gstride) {
    unsigned k[NE];
    unsigned rem = unit / p.lastq;
    const unsigned kl0 = (unit - rem * p.lastq) * 4u;
    const unsigned outer_lin = rem;
    long long base = (long long)kl0;
#pragma unroll
    for (int d = NE - 2; d >= 0; --d) {
      if (d == 0 && p.row_axis) {
        k[d] = p.row_begin + rem * p.row_step;
      } else {
        const unsigned q = rem / p.rs[d];
        k[d] = rem - q * p.rs[d];
        rem = q;
      }
      base += (long long)k[d] * p.bstr[d];
    }
    double total[4] = {0.0, 0.0, 0.0, 0.0}, inner[4] = {0.0, 0.0, 0.0, 0.0};
    bool open = false;
#pragma unroll
    for (int t = 0; t < NT; t++) {
      if (t < p.nt) {
        if (p.group_start[t]) {
          if (open) {
#pragma unroll
            for (int i = 0; i < 4; i++) total[i] = __dadd_rn(total[i], inner[i]);
          }
#pragma unroll
          for (int i = 0; i < 4; i++) inner[i] = 0.0;
          open = true;
#pragma unroll
          for (int d = 0; d < NE - 1; d++) open = open && (k[d] - (unsigned)p.m[t][d]) < p.big[d];   // unsigned: k >= m too
        }
        if (open) {
          const unsigned ml = p.m[t][NE - 1];
          const double* src = p.bigp + (base - p.delta[t]);
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const unsigned kk = kl0 + i;
            if (kk < rl && (kk - ml) < bl) inner[i] = __dadd_rn(inner[i], __dmul_rn(src[i], sv[t]));
          }
        }
      }
    }
    double* dst = p.out + (size_t)outer_lin * rl + kl0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (open) total[i] = __dadd_rn(total[i], inner[i]);
      if (kl0 + i < rl) dst[i] = total[i];
    }
  }
}

// Returns false if the product is not a stencil case (then the caller falls back to the reference-order kernel).
static bool launch_mul_stencil(Ctx& ctx, const MulArgs& a) {
  const int nd = a.ndim;
  if (a.accumulate || !a.rows.empty() || nd == 0 || nd > MAXD) return false;
  const u64 nx = prod(a.xs), ny = prod(a.ys);
  const bool small_is_x = nx <= ny;
  const Shape& ss = small_is_x ? a.xs : a.ys;
  const Shape& bs = small_is_x ? a.ys : a.xs;
  const u64 ns = std::min(nx, ny), nb = std::max(nx, ny);
  if (ns == 0 || ns > (u64)ST_MAXT || nb < 4096) return false;
  u64 row_elems = 1;
  for (int i = 1; i < nd; i++) row_elems *= a.rs[i];
  const u64 row_count = a.rs[0] == 1 ? 1 : a.row_count;
  const u64 total = row_count * row_elems;
  if (total == 0 || total >= (1ull << 32) - 65536 || a.row_begin + a.row_count * a.row_step >= (1ull << 32)) return false;
  for (int d = 0; d < nd; d++)
    if (ss[d] > 255) return false;
  // The row-staged bulk-copy kernel (kernels_horner.cu) wins inside the fused Horner loop (0.138 s against 0.202 s on
  // population_50_3vars --limit 300) but not on a single product, where the four-coefficient gather below is 2x faster
  // (0.139 ms against 0.269 ms on [297,282,297] x [2,1,2], profiles/r02_stencil_ab.txt): opt-in for A/B measurements.
  if ((ctx.bulk_products || ctx.direct_products) && launch_stencil_rows(ctx, a)) return true;
  StencilP p;
  memset(&p, 0, sizeof(p));
  Shape sst(nd, 1), bst(nd, 1);
  for (int i = nd - 2; i >= 0; --i) {
    sst[i] = sst[i + 1] * ss[i + 1];
    bst[i] = bst[i + 1] * bs[i + 1];
  }
  std::vector<int> eff;   // effective (non-unit result) axes
  for (int d = 0; d < nd; d++) {
    if (a.rs[d] == 1) {
      if (d == 0 && !(a.row_count <= 1 && a.row_begin == 0)) return false;
      // operands longer than a unit result axis never come from the operator surface (they are truncated to the
      // result degrees first); the reference's flattened 1-d leaf gives such shapes a meaning of their own
      if (a.xs[d] != 1 || a.ys[d] != 1) return false;
      continue;
    }
    eff.push_back(d);
  }
  if (eff.empty() || (int)eff.size() > MUL_MAXE) return false;
  const int ne = (int)eff.size();
  p.ne = ne;
  p.row_axis = eff[0] == 0 ? 1 : 0;
  for (int e = 0; e < ne; e++) {
    p.rs[e] = (unsigned)a.rs[eff[e]];
    p.big[e] = (unsigned)bs[eff[e]];
    p.bstr[e] = (long long)bst[eff[e]];
  }
  // the small operand's coefficients that can contribute (index 0 on every unit result axis), in visiting order:
  // ascending X index <=> ascending m if the small operand is X, descending m if it is Y
  struct Term { std::vector<unsigned> m; u64 idx; };
  std::vector<Term> terms;
  for (u64 lin = 0; lin < ns; lin++) {
    u64 rem = lin;
    std::vector<unsigned> full(nd);
    for (int d = nd - 1; d >= 0; --d) {
      full[d] = (unsigned)(rem % ss[d]);
      rem /= ss[d];
    }
    bool ok = true;
    for (int d = 0; d < nd; d++)
      if (a.rs[d] == 1 && full[d] != 0) ok = false;
    if (!ok) continue;
    Term t;
    t.idx = lin;
    for (int e = 0; e < ne; e++) t.m.push_back(full[eff[e]]);
    terms.push_back(t);
  }
  if (terms.empty()) return false;
  std::sort(terms.begin(), terms.end(), [&](const Term& x, const Term& y) { return small_is_x ? x.m < y.m : x.m > y.m; });
  p.nt = (int)terms.size();
  for (int t = 0; t < p.nt; t++) {
    long long delta = 0;
    for (int e = 0; e < ne; e++) {
      p.m[t][e] = (unsigned char)terms[t].m[e];
      delta += (long long)terms[t].m[e] * p.bstr[e];
    }
    p.delta[t] = delta;
    p.sidx[t] = (unsigned short)terms[t].idx;
    bool new_group = t == 0;
    for (int e = 0; e < ne - 1 && !new_group; e++) new_group = terms[t].m[e] != terms[t - 1].m[e];
    p.group_start[t] = new_group ? 1 : 0;
  }
  p.row_begin = (unsigned)a.row_begin;
  p.row_step = (unsigned)a.row_step;
  p.total = (unsigned)total;
  p.bigp = small_is_x ? a.y : a.x;
  p.smallp = small_is_x ? a.x : a.y;
  p.out = a.out;
  const int block = 256;
  const int grid = (int)std::max<u64>(1, std::min<u64>((total + block - 1) / block, (u64)ctx.sm_count * 32));
  const int bucket = p.nt <= 2 ? 2 : p.nt <= 4 ? 4 : p.nt <= 8 ? 8 : p.nt <= 16 ? 16 : 32;
  if (ne >= 2 && p.rs[ne - 1] >= 8 && p.bstr[ne - 1] == 1 && ctx.stencil_v4) {
    p.lastq = (p.rs[ne - 1] + 3) / 4;
    const u64 units = (total / p.rs[ne - 1]) * p.lastq;
    p.total = (unsigned)units;
    const int gridv = (int)std::max<u64>(1, std::min<u64>((units + block - 1) / block, (u64)ctx.sm_count * 32));
#define CASE_NT(N, T) case T: GTP_LAUNCH(ctx, (k_mul_stencil_v4<N, T>), gridv, block, 0, p); break;
#define CASE(N) case N: switch (bucket) { CASE_NT(N, 2) CASE_NT(N, 4) CASE_NT(N, 8) CASE_NT(N, 16) CASE_NT(N, 32) } break;
    switch (ne) {
      CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
    }
#undef CASE
#undef CASE_NT
    return true;
  }
#define CASE_NT(N, T) case T: GTP_LAUNCH(ctx, (k_mul_stencil<N, T>), grid, block, 0, p); break;
#define CASE(N) case N: switch (bucket) { CASE_NT(N, 2) CASE_NT(N, 4) CASE_NT(N, 8) CASE_NT(N, 16) CASE_NT(N, 32) } break;
  switch (ne) {
    CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
  }
#undef CASE
#undef CASE_NT
  return true;
}

// ------------------------------------------------------------------------------------------
// Shape cliff: the DFMA kernels want the last axis equal in X, Y and Z and a multiple of an even chunk (8..16); the sliding
// kernel also equal, even / multiple-of-4 plane and row counts.  Evaluation cubes have edge limit + 1 + sum(orders)
// (generating_function.rs:628-657, 756-763) -- 27, 31, 17 ... -- and used to fall to the reference-order kernel (~0.15
// TFLOP/s, 160x slower).  Zero-extending the operands to the next supported extents does not change any coefficient of
// the truncated product (absent coefficients ARE zeros, multivariate_taylor.rs:15-18), so such products are padded (two
// gather passes), multiplied by the DFMA kernels and cropped (one pass): three HBM passes against a compute-bound
// product, at the price of the padded multiply-adds (bounded below).
// ------------------------------------------------------------------------------------------
static u64 pad_chunkable(u64 l) {
  for (u64 c = l;; c++)
    if (dfma_chunk(c)) return c;
}
// 0: no padded plan; 2 / 3: zero-extend and run the blocked / sliding kernel on `best`
static int pad_plan(const Ctx& ctx, const MulArgs& a, MulArgs* out_best) {
  const int nd = a.ndim;
  if (nd < 3 || a.accumulate || !ctx.use_pad) return 0;
  const double macs = args_macs(a);
  if (macs < 4.0 * DFMA_MIN_MACS) return 0;
  auto padded = [&](bool slide) {
    MulArgs m = a;
    m.rs[nd - 1] = pad_chunkable(a.rs[nd - 1]);
    m.xs[nd - 1] = m.ys[nd - 1] = m.rs[nd - 1];
    if (slide) {
      m.rs[nd - 2] = (a.rs[nd - 2] + 3) / 4 * 4;
      m.rs[nd - 3] = (a.rs[nd - 3] + 1) / 2 * 2;
      m.xs[nd - 2] = m.ys[nd - 2] = m.rs[nd - 2];
      m.xs[nd - 3] = m.ys[nd - 3] = m.rs[nd - 3];
    }
    return m;
  };
  MulArgs best;
  int kind = 0;
  if (nd >= 4 && ctx.use_slide) {
    MulArgs m = padded(true);
    // (the sliding kernel runs ~1.4x faster per MAC than the blocked one: it wins up to ~2x padded work against the
    // blocked kernel's last-axis-only padding -- 5 x 17: planes 18, rows 20, last axis 20 = 1.99x the MACs)
    if (slide_mul_applicable(ctx, m) && args_macs(m) <= 2.05 * macs) { best = m; kind = 3; }
  }
  if (!kind) {
    MulArgs m = padded(false);
    if (blk_mul_applicable(ctx, m) && args_macs(m) <= 2.5 * macs) { best = m; kind = 2; }
  }
  if (kind) *out_best = best;
  return kind;
}
static bool launch_mul_padded(Ctx& ctx, const MulArgs& a) {
  const int nd = a.ndim;
  MulArgs best;
  const int kind = pad_plan(ctx, a, &best);
  if (!kind) return false;
  auto tail_elems = [&](const Shape& s) { u64 p = 1; for (int d = 1; d < nd; d++) p *= s[d]; return p; };
  const u64 rows = a.rows.empty() ? a.row_count : a.rows.size();
  if (prod(best.xs) >= (1ull << 32) - 4096 || prod(best.ys) >= (1ull << 32) - 4096 || rows * tail_elems(best.rs) >= (1ull << 32) - 4096) return false;
  auto pad_operand = [&](const double* src, const Shape& from, const Shape& to) -> BufP {
    if (from == to) return BufP();
    BufP b = ctx.alloc(prod(to));
    GTP_CUDA(cudaMemsetAsync(b->d, 0, prod(to) * sizeof(double), ctx.stream));
    EwOperand A;
    A.p = src;
    A.shape = from;
    launch_ew(ctx, EW_COPY, from, A, nullptr, b->d, to, {});
    return b;
  };
  BufP xp = pad_operand(a.x, a.xs, best.xs), yp = pad_operand(a.y, a.ys, best.ys);
  Shape zrows_p = best.rs, zrows = a.rs;
  zrows_p[0] = rows;
  zrows[0] = rows;
  BufP zp = ctx.alloc(prod(zrows_p));
  best.x = xp ? xp->d : a.x;
  best.y = yp ? yp->d : a.y;
  best.out = zp->d;
  if (kind == 3) launch_mul_slide(ctx, best);
  else launch_mul_blk(ctx, best);
  EwOperand Z;   // crop: the leading box of the padded rows
  Z.p = zp->d;
  Z.shape = zrows_p;
  launch_ew(ctx, EW_COPY, zrows, Z, nullptr, a.out, zrows, {});
  return true;
}

void launch_mul(Ctx& ctx, const MulArgs& a_in) {
  MulArgs a = a_in;
  if (!a.rows.empty()) {
    a.row_count = a.rows.size();
    a.row_begin = a.rows[0];
    a.row_step = 1;
  }
  const int kind = mul_kernel_kind(ctx, a);
  if (ctx.hist) {   // GTP_LAUNCH_HIST=1: log every product above 10^6 MACs (shape census of real programs)
    const double macs = args_macs(a);
    if (macs >= 1e6) {
      auto sh = [](const Shape& v) { std::string t; for (u64 x : v) t += std::to_string(x) + ","; return t; };
      fprintf(stderr, "[gtp mul] kind %d macs %.3g x [%s] y [%s] r [%s] rows %llu\n", kind, macs, sh(a.xs).c_str(), sh(a.ys).c_str(),
              sh(a.rs).c_str(), (unsigned long long)a.row_count);
    }
  }
  if (kind == 2) {
    launch_mul_blk(ctx, a);
    return;
  }
  if (kind == 3) {
    launch_mul_slide(ctx, a);
    return;
  }
  if (ctx.fast_mul && ctx.use_stencil && launch_mul_stencil(ctx, a)) return;   // bit-exact, HBM-bound small-operand products
  if (ctx.fast_mul && ctx.use_axis && launch_mul_axis(ctx, a)) return;         // bit-exact, 1-d operand x N-d tensor
  if (ctx.fast_mul && launch_mul_padded(ctx, a)) return;                       // odd extents: zero-extend, DFMA kernels, crop
  if (a.rows.empty()) {
    launch_mul_ordered(ctx, a);
    return;
  }
  // the reference-order kernel walks arithmetic progressions: one launch per maximal run of the list
  u64 row_elems = 1;
  for (int i = 1; i < a.ndim; i++) row_elems *= a.rs[i];
  size_t i = 0;
  while (i < a.rows.size()) {
    size_t j = i + 1;
    u64 step = 1;
    if (j < a.rows.size() && a.rows[j] > a.rows[i]) {
      step = a.rows[j] - a.rows[i];
      while (j + 1 < a.rows.size() && a.rows[j + 1] > a.rows[j] && a.rows[j + 1] - a.rows[j] == step) j++;
      j++;
    }
    MulArgs seg = a;
    seg.rows.clear();
    seg.row_begin = a.rows[i];
    seg.row_step = step;
    seg.row_count = j - i;
    seg.out = a.out + i * row_elems;
    launch_mul_ordered(ctx, seg);
    i = j;
  }
}

// ------------------------------------------------------------------------------------------
// FP64 pipe probes: the denominators of the product roofline, measured not quoted.
//   kind 0: DFMA, 8 independent chains per thread, every SM saturated
//   kind 1: DMMA  mma.sync.aligned.m8n8k4.f64, 4 independent accumulator tiles per warp
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_probe_dfma(int iters, double seed, double* sink) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
#pragma unroll 8
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 12345.678) sink[0] = s;
}
__global__ void __launch_bounds__(256) k_probe_dmma(int iters, double seed, double* sink) {
  double a = seed + (threadIdx.x & 31) * 1e-3, b = 1.0 + (threadIdx.x & 7) * 1e-6;
  double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
  for (int i = 0; i < iters; i++) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(e0), "+d"(e1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(f0), "+d"(f1) : "d"(a), "d"(b));
  }
  double s = c0 + c1 + d0 + d1 + e0 + e1 + f0 + f1;
  if (s == 12345.678) sink[0] = s;
}

// kind 2/4: the register row-convolution pattern of the tiled kernel (z[k] += x[j]*y[k-j], 136 DFMA,
//           operands resident in registers, nothing else in the loop) at 16 / 8 warps per SM
// kind 3/5: the 2x2-blocked pattern (544 DFMA into 3 accumulator rows) at 8 / 12 warps per SM
// They bound what ANY schedule of this arithmetic can reach on the FP64 pipe (register-file operand
// bandwidth included), separately from shared-memory and control overheads.
__global__ void __launch_bounds__(128) k_probe_rowconv(int iters, const double* __restrict__ src, double* sink) {
  extern __shared__ double dummy_smem[];
  double x[16], y[16], z[16];
#pragma unroll
  for (int i = 0; i < 16; i++) {
    x[i] = src[(threadIdx.x + i) & 63];
    y[i] = src[(threadIdx.x + 2 * i + 1) & 63];
    z[i] = 0.0;
  }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int j = 0; j < 16; j++)
#pragma unroll
      for (int k = j; k < 16; k++) z[k] = fma(x[j], y[k - j], z[k]);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; i++) s += z[i];
  if (s == 12345.678) sink[0] = s + dummy_smem[0];
}
__global__ void __launch_bounds__(128) k_probe_block22(int iters, const double* __restrict__ src, double* sink) {
  extern __shared__ double dummy_smem[];
  double xa[16], xb[16], y0[16], y1[16], z0[16], z1[16], z2[16];
#pragma unroll
  for (int i = 0; i < 16; i++) {
    xa[i] = src[(threadIdx.x + i) & 63];
    xb[i] = src[(threadIdx.x + 3 * i + 2) & 63];
    y0[i] = src[(threadIdx.x + 2 * i + 1) & 63];
    y1[i] = src[(threadIdx.x + 5 * i + 3) & 63];
    z0[i] = z1[i] = z2[i] = 0.0;
  }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int j = 0; j < 16; j++)
#pragma unroll
      for (int k = j; k < 16; k++) {
        z0[k] = fma(xa[j], y0[k - j], z0[k]);
        z1[k] = fma(xa[j], y1[k - j], z1[k]);
        z1[k] = fma(xb[j], y0[k - j], z1[k]);
        z2[k] = fma(xb[j], y1[k - j], z2[k]);
      }
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; i++) s += z0[i] + z1[i] + z2[i];
  if (s == 12345.678) sink[0] = s + dummy_smem[0];
}

void fp64_peak_probe(Ctx& ctx, int kind, int iters, double* flops, double* ms) {
  BufP sink = ctx.alloc(64);
  GTP_CUDA(cudaMemsetAsync(sink->d, 0, 64 * sizeof(double), ctx.stream));
  int grid = ctx.sm_count * 8, block = 256;
  size_t smem = 0;
  if (kind >= 2) {
    block = 128;
    int ctas_per_sm = (kind == 2) ? 4 : (kind == 5 ? 3 : 2);
    smem = (size_t)(220 * 1024 / ctas_per_sm) & ~(size_t)1023;  // dynamic smem only to pin the occupancy
    grid = ctx.sm_count * ctas_per_sm;
    GTP_CUDA(cudaFuncSetAttribute(k_probe_rowconv, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
    GTP_CUDA(cudaFuncSetAttribute(k_probe_block22, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  }
  cudaEvent_t e0, e1;
  GTP_CUDA(cudaEventCreate(&e0));
  GTP_CUDA(cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; rep++) {  // first pass warms up
    GTP_CUDA(cudaEventRecord(e0, ctx.stream));
    if (kind == 0) GTP_LAUNCH(ctx, k_probe_dfma, grid, block, 0, iters, 1.0, sink->d);
    else if (kind == 1) GTP_LAUNCH(ctx, k_probe_dmma, grid, block, 0, iters, 1.0, sink->d);
    else if (kind == 2 || kind == 4) GTP_LAUNCH(ctx, k_probe_rowconv, grid, block, smem, iters, sink->d, sink->d);
    else GTP_LAUNCH(ctx, k_probe_block22, grid, block, smem, iters, sink->d, sink->d);
    GTP_CUDA(cudaEventRecord(e1, ctx.stream));
    GTP_CUDA(cudaEventSynchronize(e1));
  }
  float t = 0;
  GTP_CUDA(cudaEventElapsedTime(&t, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  double threads = (double)grid * block;
  double f;
  if (kind == 0) f = threads * (double)iters * 8.0 * 2.0;
  else if (kind == 1) f = (threads / 32.0) * (double)iters * 4.0 * (8.0 * 8.0 * 4.0) * 2.0;
  else if (kind == 2 || kind == 4) f = threads * (double)iters * 136.0 * 2.0;
  else f = threads * (double)iters * 544.0 * 2.0;
  *ms = t;
  *flops = f / (t * 1e-3);
}

}  // namespace gtp
