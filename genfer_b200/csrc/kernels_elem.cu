// Element-wise, gather, shift and axis-reduction kernels (HBM-bound family, SURVEY 8a rows a3-a6,
// a8, a13-a16, a18).  All arithmetic is plain IEEE double with explicit __dmul_rn/__dadd_rn where
// the reference does a separate multiply and add, so these paths are bit-identical to the oracle.
#include <atomic>

#include "kernels.cuh"

namespace gtp {

// ------------------------------------------------------------------------------------------
// generic N-D element-wise kernel
// ------------------------------------------------------------------------------------------
template <int OP>
__global__ void __launch_bounds__(256) k_ew(const EwParams p) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 lin = (u64)blockIdx.x * blockDim.x + threadIdx.x; lin < p.total; lin += stride) {
    u64 rem = lin;
    long long ao = p.a_base, bo = p.b_base, oo = p.o_base;
    bool a_ok = true, b_ok = true;
    unsigned fidx = 0;
    bool first = (lin == 0);
#pragma unroll 1
    for (int d = p.ndim - 1; d >= 0; --d) {
      unsigned e = p.ext[d];
      unsigned i = (unsigned)(rem % e);
      rem /= e;
      ao += (long long)i * p.a_str[d];
      bo += (long long)i * p.b_str[d];
      oo += (long long)i * p.o_str[d];
      a_ok &= i < p.a_ext[d];
      b_ok &= i < p.b_ext[d];
      if (d == p.fax) fidx = i;
    }
    double r;
    const double sv = (OP == EW_SCALE_DEV || OP == EW_DIV_DEV || OP == EW_ADD_FIRST || OP == EW_SUB_FIRST || OP == EW_RSUB_FIRST)
                          ? (p.s ? *p.s : p.s_val) : 0.0;
    if (OP == EW_COPY) {
      double a = p.a[ao];
      r = p.fac ? __dmul_rn(a, p.fac[fidx]) : a;
    } else if (OP == EW_ADD || OP == EW_SUB) {
      r = 0.0;
      if (a_ok) r = __dadd_rn(r, p.a[ao]);
      if (b_ok) r = (OP == EW_ADD) ? __dadd_rn(r, p.b[bo]) : __dsub_rn(r, p.b[bo]);
    } else if (OP == EW_MASK) {
      r = p.keep[fidx] ? p.a[ao] : 0.0;
    } else if (OP == EW_SCALE_DEV) {
      r = __dmul_rn(sv, p.a[ao]);
    } else if (OP == EW_DIV_DEV) {
      r = __ddiv_rn(p.a[ao], sv);
    } else if (OP == EW_NEG) {
      r = -p.a[ao];
    } else if (OP == EW_ADD_FIRST) {
      r = first ? __dadd_rn(p.a[ao], sv) : p.a[ao];
    } else if (OP == EW_SUB_FIRST) {
      r = first ? __dsub_rn(p.a[ao], sv) : p.a[ao];
    } else {  // EW_RSUB_FIRST
      r = -(first ? __dsub_rn(p.a[ao], sv) : p.a[ao]);
    }
    p.out[oo] = r;
  }
}

// Fast variant (every tensor with fewer than 2^32 box elements): 32-bit index arithmetic, four independent elements per
// thread and iteration (all loads issued before the first store: the one-element loop above keeps a single 8-byte load
// in flight per thread and reaches ~64 % of HBM on a plain copy), and -- when the innermost axis is contiguous, even
// and 16-byte aligned in every tensor (VEC2) -- 16-byte loads and stores.  `tab` is a factor table passed in the
// kernel parameters (host-built derivative / binomial factors: no table-building launch); fac == nullptr, tab == nullptr:
// no factor.  Arithmetic is identical to k_ew.
constexpr int FAC_TAB = 1024;   // 8 KB of kernel parameters (large parameter space, CUDA >= 12.1)
struct FacTab {
  double f[FAC_TAB];
};
template <int OP, bool VEC2>
__device__ __forceinline__ void ew_fast_body(const EwParams& p, const double* __restrict__ fac) {
  constexpr int U = 4;
  const unsigned units = (unsigned)p.total;   // elements, or element pairs along the innermost axis (VEC2)
  const unsigned step = blockDim.x * U;
  for (unsigned base = blockIdx.x * step + threadIdx.x; base < units; base += gridDim.x * step) {
    long long ao[U], bo[U], oo[U];
    bool a_ok[U], b_ok[U], live[U];
    unsigned fidx[U];
#pragma unroll
    for (int j = 0; j < U; j++) {
      const unsigned lin = base + j * blockDim.x;
      live[j] = lin < units;
      unsigned rem = live[j] ? lin : 0u;
      ao[j] = p.a_base;
      bo[j] = p.b_base;
      oo[j] = p.o_base;
      a_ok[j] = b_ok[j] = true;
      fidx[j] = 0;
#pragma unroll 1
      for (int d = p.ndim - 1; d >= 0; --d) {
        const unsigned e = p.ext[d];
        const unsigned q = rem / e, i = rem - q * e;
        rem = q;
        const unsigned ii = (VEC2 && d == p.ndim - 1) ? 2u * i : i;
        ao[j] += (long long)ii * p.a_str[d];
        bo[j] += (long long)ii * p.b_str[d];
        oo[j] += (long long)ii * p.o_str[d];
        a_ok[j] &= ii < p.a_ext[d];
        b_ok[j] &= ii < p.b_ext[d];
        if (d == p.fax) fidx[j] = ii;
      }
    }
    double2 av[U], bv[U];
    constexpr bool READS_A_ALWAYS = !(OP == EW_ADD || OP == EW_SUB);
    constexpr bool READS_B = (OP == EW_ADD || OP == EW_SUB);
#pragma unroll
    for (int j = 0; j < U; j++) {
      av[j] = bv[j] = make_double2(0.0, 0.0);
      if (live[j] && (READS_A_ALWAYS || a_ok[j])) {
        if (VEC2) av[j] = *reinterpret_cast<const double2*>(p.a + ao[j]);
        else av[j].x = p.a[ao[j]];
      }
      if (READS_B && live[j] && b_ok[j]) {
        if (VEC2) bv[j] = *reinterpret_cast<const double2*>(p.b + bo[j]);
        else bv[j].x = p.b[bo[j]];
      }
    }
    double sv = 0.0;
    if (OP == EW_SCALE_DEV || OP == EW_DIV_DEV || OP == EW_ADD_FIRST || OP == EW_SUB_FIRST || OP == EW_RSUB_FIRST) sv = p.s ? *p.s : p.s_val;
#pragma unroll
    for (int j = 0; j < U; j++) {
      if (!live[j]) continue;
      const bool first = (base + j * blockDim.x) == 0;
      double2 r;
#pragma unroll
      for (int h = 0; h < (VEC2 ? 2 : 1); h++) {
        const double a = h ? av[j].y : av[j].x, b = h ? bv[j].y : bv[j].x;
        const bool f0 = first && h == 0;
        double v;
        if (OP == EW_COPY) {
          const bool last_fax = p.fax == p.ndim - 1;
          v = fac ? __dmul_rn(a, fac[fidx[j] + ((VEC2 && last_fax) ? h : 0)]) : a;
        } else if (OP == EW_ADD || OP == EW_SUB) {
          v = 0.0;
          if (a_ok[j]) v = __dadd_rn(v, a);
          if (b_ok[j]) v = (OP == EW_ADD) ? __dadd_rn(v, b) : __dsub_rn(v, b);
        } else if (OP == EW_MASK) {
          const bool last_fax = p.fax == p.ndim - 1;
          v = p.keep[fidx[j] + ((VEC2 && last_fax) ? h : 0)] ? a : 0.0;
        } else if (OP == EW_SCALE_DEV) {
          v = __dmul_rn(sv, a);
        } else if (OP == EW_DIV_DEV) {
          v = __ddiv_rn(a, sv);
        } else if (OP == EW_NEG) {
          v = -a;
        } else if (OP == EW_ADD_FIRST) {
          v = f0 ? __dadd_rn(a, sv) : a;
        } else if (OP == EW_SUB_FIRST) {
          v = f0 ? __dsub_rn(a, sv) : a;
        } else {  // EW_RSUB_FIRST
          v = -(f0 ? __dsub_rn(a, sv) : a);
        }
        if (h) r.y = v; else r.x = v;
      }
      if (VEC2) *reinterpret_cast<double2*>(p.out + oo[j]) = r;
      else p.out[oo[j]] = r.x;
    }
  }
}
template <int OP, bool VEC2>
__global__ void __launch_bounds__(256) k_ew_fast(const __grid_constant__ EwParams p) {
  ew_fast_body<OP, VEC2>(p, p.fac);
  if (p.cls.slot) cls_epilogue(p.out, p.cls.p, p.cls.slot, p.cls.seq);   // gridDim.x == 1 (launch_ew)
}
template <bool VEC2>
__global__ void __launch_bounds__(256) k_ew_tab(const __grid_constant__ EwParams p, const __grid_constant__ FacTab tab) {
  // staged in shared memory: a warp's lanes index the table with different k, and divergent constant-bank reads serialise
  __shared__ double sfac[FAC_TAB];
  for (int i = threadIdx.x; i < FAC_TAB; i += blockDim.x) sfac[i] = tab.f[i];
  __syncthreads();
  ew_fast_body<EW_COPY, VEC2>(p, sfac);
  if (p.cls.slot) cls_epilogue(p.out, p.cls.p, p.cls.slot, p.cls.seq);
}

// Two-axis gathers with contiguous rows -- what derivative / taylor_expansion_of_coeff / prefix truncations / slices become
// after axis coalescing: out[r, c] = a[a_base + r * a_row + c] * fac[r or c], `out` dense.  The generic kernel decodes every
// element's index (two divisions per element: 38-50 % of HBM on 16^6 tensors, instruction-bound); here a thread owns FOUR
// consecutive output coefficients, decodes once, walks the row boundary by compare-and-wrap, issues its four loads before the
// first store and stores 16 bytes at a time.  Arithmetic identical (one IEEE multiply or a plain copy).
struct Ew2dParams {
  const double* a;
  double* out;
  unsigned long long total;      // rows * cols
  unsigned cols;
  long long a_row;               // source stride between rows
  int fax;                       // 0: factor indexed by the row, 1: by the column, -1: none
  FusedClsArgs cls;
};
template <bool TAB>
__global__ void __launch_bounds__(256) k_ew2d(const __grid_constant__ Ew2dParams p, const __grid_constant__ FacTab tab) {
  __shared__ double sfac[TAB ? FAC_TAB : 1];
  if (TAB) {
    for (int i = threadIdx.x; i < FAC_TAB; i += blockDim.x) sfac[i] = tab.f[i];
    __syncthreads();
  }
  const unsigned long long nq = (p.total + 3ull) / 4ull;
  for (unsigned long long qd = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; qd < nq; qd += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long o0 = qd * 4ull;
    unsigned long long r;
    unsigned c;
    if (p.total <= 0xffffffffull) {   // 32-bit division: the 64-bit one costs more instructions than the rest of the thread's work
      const unsigned o32 = (unsigned)o0, r32 = o32 / (unsigned)p.cols;
      r = r32;
      c = o32 - r32 * (unsigned)p.cols;
    } else {
      r = o0 / p.cols;
      c = (unsigned)(o0 - r * p.cols);
    }
    double v[4];
    unsigned fi[4];
    bool live[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      live[j] = o0 + j < p.total;
      v[j] = live[j] ? p.a[(long long)r * p.a_row + c] : 0.0;
      fi[j] = p.fax == 0 ? (unsigned)r : c;
      if (++c == p.cols) { c = 0; r++; }
    }
    if (TAB) {
#pragma unroll
      for (int j = 0; j < 4; j++) v[j] = __dmul_rn(v[j], sfac[fi[j]]);
    }
    double* dst = p.out + o0;
    if (live[3]) {
      *reinterpret_cast<double2*>(dst) = make_double2(v[0], v[1]);
      *reinterpret_cast<double2*>(dst + 2) = make_double2(v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (live[j]) dst[j] = v[j];
    }
  }
  if (p.cls.slot) cls_epilogue(p.out, p.cls.p, p.cls.slot, p.cls.seq);
}

bool fused_cls_begin(Ctx& ctx, const double* out, const Shape& shape, FusedClsArgs* f) {
  f->slot = nullptr;
  const u64 total = prod(shape);
  if (!ctx.cls_ring || total == 0 || total > 1024 || shape.size() > (size_t)MAXD) return false;
  const unsigned long long seq = ++ctx.cls_seq;
  f->slot = ctx.cls_ring + (seq % Ctx::CLS_RING);
  f->seq = seq;
  ClsParams& p = f->p;
  memset(&p, 0, sizeof(p));
  p.ndim = (int)shape.size();
  p.total = total;
  long long st = 1;
  for (int d = p.ndim - 1; d >= 0; --d) {
    p.shape[d] = (unsigned)shape[d];
    p.str[d] = st;
    st *= (long long)shape[d];
  }
  p.all_mask = p.ndim >= 32 ? 0xffffffffu : ((1u << p.ndim) - 1u);
  FusedCls& e = ctx.fused_cls[out];
  e.seq = seq;
  e.shape = shape;
  return true;
}

static Shape strides_of(const Shape& shape) {
  Shape st(shape.size(), 1);
  for (int i = (int)shape.size() - 2; i >= 0; --i) st[i] = st[i + 1] * shape[i + 1];
  return st;
}

void launch_ew(Ctx& ctx, EwOp op, const Shape& box, const EwOperand& a, const EwOperand* b, double* out,
               const Shape& out_shape, const Shape& out_lo, int fax, const double* fac,
               const unsigned char* keep, const double* s, const double* tab, int tab_len, const double* s_host) {
  const int nd = (int)box.size();
  GTP_CHECK(nd <= MAXD, GTP_ERR_ARG, "ndim exceeds GTP_MAX_NDIM");
  u64 total = prod(box);
  if (total == 0) return;
  // per-axis description
  struct Ax {
    u64 ext, a_ext, b_ext;
    long long a_str, b_str, o_str;
    bool special;
  };
  std::vector<Ax> ax(nd);
  Shape ast = strides_of(a.shape), ost = strides_of(out_shape), bst;
  if (b) bst = strides_of(b->shape);
  long long a_base = 0, b_base = 0, o_base = 0;
  for (int d = 0; d < nd; d++) {
    ax[d].ext = box[d];
    ax[d].a_ext = a.valid.empty() ? box[d] : std::min<u64>(a.valid[d], box[d]);
    ax[d].b_ext = (b && !b->valid.empty()) ? std::min<u64>(b->valid[d], box[d]) : box[d];
    ax[d].a_str = (long long)ast[d];
    ax[d].b_str = b ? (long long)bst[d] : 0;
    ax[d].o_str = (long long)ost[d];
    ax[d].special = (d == fax);
    a_base += (long long)(a.lo.empty() ? 0 : a.lo[d]) * (long long)ast[d];
    if (b) b_base += (long long)(b->lo.empty() ? 0 : b->lo[d]) * (long long)bst[d];
    o_base += (long long)(out_lo.empty() ? 0 : out_lo[d]) * (long long)ost[d];
  }
  // drop unit axes, then merge axis d+1 into d when the pair is contiguous in every tensor and
  // fully valid (so validity / factor indexing is unaffected)
  std::vector<Ax> c;
  for (int d = 0; d < nd; d++)
    if (ax[d].ext != 1 || ax[d].special) c.push_back(ax[d]);
  if (c.empty()) c.push_back(Ax{1, 1, 1, 0, 0, 0, false});
  for (size_t d = c.size(); d-- > 1;) {
    Ax& hi = c[d - 1];
    Ax& lo = c[d];
    bool full = lo.a_ext == lo.ext && lo.b_ext == lo.ext && hi.a_ext == hi.ext && hi.b_ext == hi.ext;
    bool contig = hi.a_str == lo.a_str * (long long)lo.ext && hi.o_str == lo.o_str * (long long)lo.ext &&
                  (!b || hi.b_str == lo.b_str * (long long)lo.ext);
    if (full && contig && !hi.special && !lo.special && hi.ext * lo.ext < (1ull << 31)) {
      hi.ext *= lo.ext;
      hi.a_ext = hi.b_ext = hi.ext;
      hi.a_str = lo.a_str;
      hi.b_str = lo.b_str;
      hi.o_str = lo.o_str;
      c.erase(c.begin() + d);
    }
  }
  EwParams p;
  memset(&p, 0, sizeof(p));
  p.ndim = (int)c.size();
  p.fax = -1;
  p.total = total;
  for (int d = 0; d < p.ndim; d++) {
    GTP_CHECK(c[d].ext < (1ull << 32), GTP_ERR_ARG, "axis too long");
    p.ext[d] = (unsigned)c[d].ext;
    p.a_ext[d] = (unsigned)c[d].a_ext;
    p.b_ext[d] = b ? (unsigned)c[d].b_ext : 0;
    p.a_str[d] = c[d].a_str;
    p.b_str[d] = c[d].b_str;
    p.o_str[d] = c[d].o_str;
    if (c[d].special) p.fax = d;
  }
  p.a_base = a_base;
  p.b_base = b_base;
  p.o_base = o_base;
  p.a = a.p;
  p.b = b ? b->p : nullptr;
  p.out = out;
  p.fac = fac;
  p.keep = keep;
  p.s = s_host ? nullptr : s;
  p.s_val = s_host ? *s_host : 0.0;
  int block = 256;
  // two-axis copy / scale with contiguous rows and a dense output: four consecutive coefficients per thread
  // (a single contiguous run keeps the 16-byte path below)
  if (op == EW_COPY && !b && !fac && p.ndim == 2 && total >= 4096 && total < (1ull << 40) &&
      p.a_str[p.ndim - 1] == 1 && p.o_str[p.ndim - 1] == 1 && p.a_ext[p.ndim - 1] == p.ext[p.ndim - 1] &&
      (p.ndim == 1 || (p.o_str[0] == (long long)p.ext[1] && p.a_ext[0] == p.ext[0])) &&
      (reinterpret_cast<uintptr_t>(out + o_base) & 15u) == 0 && (!tab || tab_len <= FAC_TAB)) {
    Ew2dParams q;
    memset(&q, 0, sizeof(q));
    q.a = a.p + a_base;
    q.out = out + o_base;
    q.total = total;
    q.cols = p.ndim == 2 ? p.ext[1] : p.ext[0];
    q.a_row = p.ndim == 2 ? p.a_str[0] : (long long)p.ext[0];
    q.fax = !tab ? -1 : (p.ndim == 2 ? p.fax : 1);
    if (!(tab && p.fax < 0)) {
      const u64 nq = (total + 3) / 4;
      const int grid = (int)std::max<u64>(1, std::min<u64>((nq + block - 1) / block, (u64)ctx.sm_count * 16));
      bool whole = box == out_shape;
      for (u64 l0 : out_lo) whole = whole && l0 == 0;
      if (whole && grid == 1) fused_cls_begin(ctx, out, out_shape, &q.cls);
      FacTab t;
      if (tab) {
        memcpy(t.f, tab, sizeof(double) * tab_len);
        GTP_LAUNCH(ctx, k_ew2d<true>, grid, block, 0, q, t);
      } else {
        GTP_LAUNCH(ctx, k_ew2d<false>, grid, block, 0, q, t);
      }
      return;
    }
  }
  if (total < (1ull << 32) - 4096) {
    // innermost axis contiguous, even and 16-byte aligned everywhere: element pairs
    const int l = p.ndim - 1;
    auto even_off = [&](long long base, const long long* str, const double* ptr) {
      if (!ptr) return true;
      if ((reinterpret_cast<uintptr_t>(ptr) & 15u) || (base & 1)) return false;
      for (int d = 0; d < l; d++)
        if (str[d] & 1) return false;
      return str[l] == 1;
    };
    bool vec2 = (p.ext[l] % 2 == 0) && (p.a_ext[l] % 2 == 0) && (!b || p.b_ext[l] % 2 == 0) &&
                even_off(p.a_base, p.a_str, p.a) && even_off(p.o_base, p.o_str, p.out) && (!b || even_off(p.b_base, p.b_str, p.b));
    if (vec2) {
      p.ext[l] /= 2;
      p.total = total / 2;
    }
    const u64 units = p.total;
    int grid = (int)std::max<u64>(1, std::min<u64>((units + block * 4 - 1) / (block * 4), (u64)ctx.sm_count * 16));
    bool whole = box == out_shape;
    for (u64 l0 : out_lo) whole = whole && l0 == 0;
    if (whole && grid == 1) fused_cls_begin(ctx, out, out_shape, &p.cls);   // the producer classifies its own output
    if (op == EW_COPY && tab) {
      FacTab t;
      memcpy(t.f, tab, sizeof(double) * tab_len);
      if (vec2) GTP_LAUNCH(ctx, k_ew_tab<true>, grid, block, 0, p, t);
      else GTP_LAUNCH(ctx, k_ew_tab<false>, grid, block, 0, p, t);
      return;
    }
    switch (op) {
#define CASE(O) case O: if (vec2) GTP_LAUNCH(ctx, (k_ew_fast<O, true>), grid, block, 0, p); else GTP_LAUNCH(ctx, (k_ew_fast<O, false>), grid, block, 0, p); break;
      CASE(EW_COPY) CASE(EW_ADD) CASE(EW_SUB) CASE(EW_MASK) CASE(EW_SCALE_DEV) CASE(EW_DIV_DEV)
      CASE(EW_NEG) CASE(EW_ADD_FIRST) CASE(EW_SUB_FIRST) CASE(EW_RSUB_FIRST)
#undef CASE
    }
    return;
  }
  GTP_CHECK(!tab, GTP_ERR_ARG, "host factor tables need the fast element-wise path");
  u64 want = (total + block - 1) / block;
  int grid = (int)std::min<u64>(want, (u64)ctx.sm_count * 16);
  switch (op) {
#define CASE(O) case O: GTP_LAUNCH(ctx, k_ew<O>, grid, block, 0, p); break;
    CASE(EW_COPY) CASE(EW_ADD) CASE(EW_SUB) CASE(EW_MASK) CASE(EW_SCALE_DEV) CASE(EW_DIV_DEV)
    CASE(EW_NEG) CASE(EW_ADD_FIRST) CASE(EW_SUB_FIRST) CASE(EW_RSUB_FIRST)
#undef CASE
  }
}

// Host-built factor tables (plain IEEE double multiplications and divisions in the reference's incremental order, so
// bit-identical to k_factors): up to 256 entries travel in the kernel parameters.
bool host_factors(int kind, u64 n, u64 len, double* fac, double m) {
  if (len > (u64)FAC_TAB || kind > 2) return false;
  if (kind == 2) {  // powers m^k (:557-565)
    volatile double f = 1.0;
    for (u64 k = 0; k < len; k++) {
      fac[k] = f;
      f = f * m;
    }
    return true;
  }
  if (kind == 0) {  // derivative :472-479
    volatile double ff = 1.0;
    for (u64 i = 1; i <= n; i++) ff = ff * (double)(unsigned)i;
    for (u64 k = 0; k < len; k++) {
      fac[k] = ff;
      volatile double q = (double)(unsigned)(n + k + 1) / (double)(unsigned)(k + 1);
      ff = ff * q;
    }
  } else {  // taylor_expansion_of_coeff :499-507
    volatile double f = 1.0;
    fac[0] = 1.0;
    for (u64 k = 1; k < len; k++) {
      volatile double q = (double)(unsigned)(n + k) / (double)(unsigned)k;
      f = f * q;
      fac[k] = f;
    }
  }
  return true;
}

// ------------------------------------------------------------------------------------------
// mul_linear (:611-623) in one pass over the (outer, len, inner) view of axis v:
//   out[o,k,i] = (0 + m x[o,k-1,i]) + c x[o,k,i]      k < xlen     (Add of `mul_var` and `self * c`, :873-880)
//              =  0 + m x[o,k-1,i]                    k == xlen    (the result is one slice longer than x)
//   c == 0:   out[o,k,i] = m x[o,k-1,i]  (mul_var alone, :589-608; slice 0 is +0)
// Same products, same additions and the same zero-extension as the reference's composition (which costs a memset and
// four more passes over HBM); x[.,k-1,.] is re-read from L1/L2.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_mul_linear(const double* __restrict__ x, double* __restrict__ out, unsigned total,
                                                   unsigned xlen, unsigned olen, unsigned inner, double c, double m, int var_only,
                                                   const __grid_constant__ FusedClsArgs cls) {
  constexpr int U = 4;
  const unsigned step = blockDim.x * U;
  for (unsigned base = blockIdx.x * step + threadIdx.x; base < total; base += gridDim.x * step) {
    double cur[U], prev[U];
    unsigned kk[U];
#pragma unroll
    for (int j = 0; j < U; j++) {
      const unsigned lin = base + j * blockDim.x;
      cur[j] = prev[j] = 0.0;
      kk[j] = 0;
      if (lin < total) {
        const unsigned q = lin / inner, i = lin - q * inner;
        const unsigned o = q / olen, k = q - o * olen;
        kk[j] = k;
        const size_t at = ((size_t)o * xlen + k) * inner + i;
        if (k < xlen && !var_only) cur[j] = x[at];
        if (k >= 1) prev[j] = x[at - inner];     // k <= xlen always (olen <= xlen + 1)
      }
    }
#pragma unroll
    for (int j = 0; j < U; j++) {
      const unsigned lin = base + j * blockDim.x;
      if (lin >= total) continue;
      const double sh = kk[j] >= 1 ? __dmul_rn(prev[j], m) : 0.0;
      double r;
      if (var_only) r = sh;
      else {
        r = __dadd_rn(0.0, sh);
        if (kk[j] < xlen) r = __dadd_rn(r, __dmul_rn(c, cur[j]));
      }
      out[lin] = r;
    }
  }
  if (cls.slot) cls_epilogue(out, cls.p, cls.slot, cls.seq);
}
void launch_mul_linear(Ctx& ctx, const double* x, double* out, u64 outer, u64 xlen, u64 olen, u64 inner, double c, double m,
                       const Shape& out_shape) {
  const u64 total = outer * olen * inner;
  if (total == 0) return;
  int grid = (int)std::max<u64>(1, std::min<u64>((total + 1023) / 1024, (u64)ctx.sm_count * 16));
  FusedClsArgs cls;
  cls.slot = nullptr;
  if (grid == 1) fused_cls_begin(ctx, out, out_shape, &cls);
  GTP_LAUNCH(ctx, k_mul_linear, grid, 256, 0, x, out, (unsigned)total, (unsigned)xlen, (unsigned)olen, (unsigned)inner, c, m,
             c == 0.0 ? 1 : 0, cls);
}

// ------------------------------------------------------------------------------------------
__global__ void k_fill(double* dst, u64 n, double v) {
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = v;
}
void launch_fill(Ctx& ctx, double* dst, u64 n, double value) {
  if (n == 0) return;
  if (value == 0.0 && !std::signbit(value)) {
    GTP_CUDA(cudaMemsetAsync(dst, 0, n * sizeof(double), ctx.stream));
    return;
  }
  int grid = (int)std::min<u64>((n + 255) / 256, (u64)ctx.sm_count * 16);
  GTP_LAUNCH(ctx, k_fill, grid, 256, 0, dst, n, value);
}

// Sequential factor tables (one thread; <= a few thousand steps): the reference builds these
// incrementally in exactly this order, so the table is bit-identical.
__global__ void k_factors(int kind, u64 n, u64 len, const double* m, double* fac) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (kind == 0) {  // derivative :472-479
    double ff = 1.0;
    for (u64 i = 1; i <= n; i++) ff = __dmul_rn(ff, (double)(unsigned)i);
    for (u64 k = 0; k < len; k++) {
      fac[k] = ff;
      ff = __dmul_rn(ff, __ddiv_rn((double)(unsigned)(n + k + 1), (double)(unsigned)(k + 1)));
    }
  } else if (kind == 1) {  // taylor_expansion_of_coeff :499-507
    double f = 1.0;
    fac[0] = 1.0;
    for (u64 k = 1; k < len; k++) {
      f = __dmul_rn(f, __ddiv_rn((double)(unsigned)(n + k), (double)(unsigned)k));
      fac[k] = f;
    }
  } else {  // powers :557-565
    double f = 1.0, mm = *m;
    for (u64 k = 0; k < len; k++) {
      fac[k] = f;
      f = __dmul_rn(f, mm);
    }
  }
}
void launch_factors(Ctx& ctx, int kind, u64 n, u64 len, const double* m, double* fac) {
  GTP_LAUNCH(ctx, k_factors, 1, 32, 0, kind, n, len, m, fac);
}

// ------------------------------------------------------------------------------------------
// shift_down.  out[o,0,i] = in[o,n,i] + sum_{a<n} in[o,a,i]   (or the plain axis sum when
// len <= n+1); out[o,a',i] = in[o,n+a',i].  Summation order follows ndarray 0.15.6 sum_axis:
//  * inner > 1  (axis is not the minimum-stride axis): res = 0; res += in[a] for a ascending
//  * inner == 1 (contiguous lanes): 8-way unrolled fold (numeric_util::unrolled_fold)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_shift_down_strided(const double* __restrict__ in, double* __restrict__ out,
                                                           u64 outer, u64 len, u64 inner, u64 n, u64 out_len) {
  // one thread per (o, i): the slices a = 0..len-1 are `inner` apart, so a warp reads 32
  // consecutive doubles of each slice (coalesced), and copies the tail slices as it goes.
  const u64 total = outer * inner;
  const u64 stride = (u64)gridDim.x * blockDim.x;
  const u64 head = (len <= n + 1) ? len : n;  // slices folded into the sum_axis part
  for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    u64 o = t / inner, i = t - o * inner;
    const double* src = in + o * len * inner + i;
    double* dst = out + o * out_len * inner + i;
    double acc = 0.0;
    u64 a = 0;
    for (; a + 4 <= head; a += 4) {  // 4 independent loads in flight
      double v0 = src[(a + 0) * inner], v1 = src[(a + 1) * inner];
      double v2 = src[(a + 2) * inner], v3 = src[(a + 3) * inner];
      acc = __dadd_rn(acc, v0);
      acc = __dadd_rn(acc, v1);
      acc = __dadd_rn(acc, v2);
      acc = __dadd_rn(acc, v3);
    }
    for (; a < head; a++) acc = __dadd_rn(acc, src[a * inner]);
    if (len <= n + 1) {
      dst[0] = acc;
    } else {
      dst[0] = __dadd_rn(src[n * inner], acc);
      for (u64 k = 1; k < out_len; k++) dst[k * inner] = src[(n + k) * inner];
    }
  }
}

// contiguous lanes: 8 threads cooperate on one lane, thread l owning p_l of unrolled_fold
__global__ void __launch_bounds__(256) k_shift_down_lanes(const double* __restrict__ in, double* __restrict__ out,
                                                         u64 outer, u64 len, u64 n, u64 out_len) {
  const u64 lanes_per_block = blockDim.x / 8;
  const unsigned l = threadIdx.x & 7;
  const unsigned full = 0xffffffffu;
  const u64 head = (len <= n + 1) ? len : n;
  for (u64 o = (u64)blockIdx.x * lanes_per_block + threadIdx.x / 8; o < (outer + lanes_per_block - 1) / lanes_per_block * lanes_per_block;
       o += (u64)gridDim.x * lanes_per_block) {
    bool active = o < outer;
    const double* src = in + (active ? o : 0) * len;
    double p = 0.0;
    u64 chunks = head / 8;
    if (active)
      for (u64 c = 0; c < chunks; c++) p = __dadd_rn(p, src[c * 8 + l]);
    // q_l = p_l + p_{l+4} for l < 4
    double hi = __shfl_down_sync(full, p, 4, 8);
    double q = __dadd_rn(p, hi);
    double q1 = __shfl_sync(full, q, 1, 8), q2 = __shfl_sync(full, q, 2, 8), q3 = __shfl_sync(full, q, 3, 8);
    if (active && l == 0) {
      double acc = 0.0;
      acc = __dadd_rn(acc, q);
      acc = __dadd_rn(acc, q1);
      acc = __dadd_rn(acc, q2);
      acc = __dadd_rn(acc, q3);
      for (u64 a = chunks * 8; a < head; a++) acc = __dadd_rn(acc, src[a]);
      double* dst = out + o * out_len;
      dst[0] = (len <= n + 1) ? acc : __dadd_rn(src[n], acc);
    }
    if (active && len > n + 1) {
      double* dst = out + o * out_len;
      for (u64 k = 1 + l; k < out_len; k += 8) dst[k] = src[n + k];
    }
  }
}

// contiguous SHORT lanes (len <= 64, the cube case): a CTA stages a tile of 256 whole lanes in shared memory with
// coalesced 16-byte loads (the tile is one contiguous span of HBM), then thread i folds lane i in exactly the
// order of the 8-threads-per-lane kernel above (p_0..p_7 strided partials, (p_l + p_{l+4}) combined in order,
// sequential tail), and the surviving slices are written back as one contiguous span.  The lane stride in
// shared memory is odd (in doubles) so the 64-bit row reads of a half-warp hit 16 distinct bank pairs.
constexpr int SD_LANES = 256;
__global__ void __launch_bounds__(SD_LANES) k_shift_down_tile(const double* __restrict__ in, double* __restrict__ out,
                                                             u64 outer, unsigned len, unsigned n, unsigned out_len, unsigned pad) {
  extern __shared__ double tile[];
  const u64 lane0 = (u64)blockIdx.x * SD_LANES;
  const unsigned lanes = (unsigned)min((u64)SD_LANES, outer - lane0);
  const double* src = in + lane0 * len;
  const unsigned total = lanes * len;
  if ((len & 1u) == 0) {   // rows hold an even number of doubles: the span is 16-byte aligned with the tensor
    const double2* src2 = reinterpret_cast<const double2*>(src);
    const unsigned half = total / 2;
    // batches of 8 independent 16-byte loads per thread before the first shared-memory store: with one load in flight
    // per thread an SM keeps only ~24 KB in flight, about a third of what HBM3e latency x bandwidth asks for
    for (unsigned e0 = threadIdx.x; e0 < half; e0 += 8 * SD_LANES) {
      double2 v[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const unsigned e = e0 + i * SD_LANES;
        if (e < half) v[i] = __ldcs(src2 + e);
      }
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const unsigned e = e0 + i * SD_LANES;
        if (e < half) {
          unsigned o = (2 * e) / len, a = 2 * e - o * len;
          tile[o * pad + a] = v[i].x;
          tile[o * pad + a + 1] = v[i].y;
        }
      }
    }
  } else {
    for (unsigned e = threadIdx.x; e < total; e += SD_LANES) {
      unsigned o = e / len, a = e - o * len;
      tile[o * pad + a] = src[e];
    }
  }
  __syncthreads();
  const unsigned head = (len <= n + 1) ? len : n;
  if (threadIdx.x < lanes) {
    double* row = tile + threadIdx.x * pad;
    double p[8];
#pragma unroll
    for (int l = 0; l < 8; l++) p[l] = 0.0;
    const unsigned chunks = head / 8;
    for (unsigned c = 0; c < chunks; c++) {
#pragma unroll
      for (int l = 0; l < 8; l++) p[l] = __dadd_rn(p[l], row[c * 8 + l]);
    }
    double acc = 0.0;
#pragma unroll
    for (int l = 0; l < 4; l++) acc = __dadd_rn(acc, __dadd_rn(p[l], p[l + 4]));
    for (unsigned a = chunks * 8; a < head; a++) acc = __dadd_rn(acc, row[a]);
    if (len <= n + 1) {                                   // the single surviving slice: coalesced direct store
      out[lane0 + threadIdx.x] = acc;
    } else {
      row[n] = __dadd_rn(row[n], acc);
    }
  }
  if (len <= n + 1) return;
  __syncthreads();
  double* dst = out + lane0 * out_len;
  for (unsigned e = threadIdx.x; e < lanes * out_len; e += SD_LANES) {
    unsigned o = e / out_len, k = e - o * out_len;
    dst[e] = tile[o * pad + n + k];
  }
}

void launch_shift_down(Ctx& ctx, const double* in, double* out, u64 outer, u64 len, u64 inner, u64 n,
                       bool last_axis) {
  u64 out_len = (len <= n + 1) ? 1 : len - n;
  if (inner > 1 || !last_axis) {
    u64 total = outer * inner;
    int grid = (int)std::max<u64>(1, std::min<u64>((total + 255) / 256, (u64)ctx.sm_count * 32));
    GTP_LAUNCH(ctx, k_shift_down_strided, grid, 256, 0, in, out, outer, len, inner, n, out_len);
  } else if (len <= 64 && outer >= 1024 && (reinterpret_cast<uintptr_t>(in) & 15u) == 0 &&
             (outer + SD_LANES - 1) / SD_LANES < (1u << 31)) {
    unsigned pad = (unsigned)((len & 1) ? len : len + 1);
    size_t smem = (size_t)SD_LANES * pad * sizeof(double);
    allow_dyn_smem(k_shift_down_tile, ctx.device, SD_LANES * 65 * 8);
    unsigned grid = (unsigned)((outer + SD_LANES - 1) / SD_LANES);
    GTP_LAUNCH(ctx, k_shift_down_tile, grid, SD_LANES, smem, in, out, outer, (unsigned)len, (unsigned)n, (unsigned)out_len, pad);
  } else {
    u64 lanes_per_block = 256 / 8;
    int grid = (int)std::max<u64>(1, std::min<u64>((outer + lanes_per_block - 1) / lanes_per_block, (u64)ctx.sm_count * 32));
    GTP_LAUNCH(ctx, k_shift_down_lanes, grid, 256, 0, in, out, outer, len, n, out_len);
  }
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sum_partial(const double* __restrict__ in, u64 n, double* partial) {
  __shared__ double sh[8];
  double acc = 0.0;
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc += in[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 8) {
    acc = sh[threadIdx.x];
    for (int o = 4; o > 0; o >>= 1) acc += __shfl_down_sync(0xffu, acc, o);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
  }
}
void launch_sum_all(Ctx& ctx, const double* in, u64 n, double* out_dev) {
  int grid = (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)ctx.sm_count * 8));
  if (grid == 1) {
    GTP_LAUNCH(ctx, k_sum_partial, 1, 256, 0, in, n, out_dev);
    return;
  }
  BufP partial = ctx.alloc(grid);
  GTP_LAUNCH(ctx, k_sum_partial, grid, 256, 0, in, n, partial->d);
  GTP_LAUNCH(ctx, k_sum_partial, 1, 256, 0, partial->d, (u64)grid, out_dev);
}

// ------------------------------------------------------------------------------------------
// classify: which axes v could be the linear axis of extract_linear (:275-294)?  A non-zero
// element at multi-index idx rules out axis v unless idx is zero everywhere except possibly
// idx[v] <= 1.  One pass builds the OR of the per-element "ruled out" masks; blocks stop early
// once every axis is ruled out (dense operands bail out after their first tile).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_classify(const double* __restrict__ in, const ClsParams p, Readback* rb) {
  __shared__ unsigned sh_mask, sh_global;
  if (threadIdx.x == 0) sh_mask = 0;
  __syncthreads();
  u64 stride = (u64)gridDim.x * blockDim.x;
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < p.total; base += stride) {
    if (threadIdx.x == 0) sh_global = *(volatile unsigned*)&rb->viol_mask;
    __syncthreads();
    if ((sh_global & p.all_mask) == p.all_mask) break;  // uniform: someone already ruled out every axis
    u64 lin = base + threadIdx.x;
    unsigned mask = 0;
    if (lin < p.total) {
      double x = in[lin];
      if (x != 0.0) {
        u64 rem = lin;
        int nz_axis = -1, nz_count = 0;
        unsigned nz_val = 0;
        for (int d = p.ndim - 1; d >= 0; --d) {
          unsigned i = (unsigned)(rem % p.shape[d]);
          rem /= p.shape[d];
          if (i != 0) {
            nz_count++;
            nz_axis = d;
            nz_val = i;
          }
        }
        if (nz_count >= 2) mask = p.all_mask;
        else if (nz_count == 1) mask = (nz_val >= 2) ? p.all_mask : (p.all_mask & ~(1u << nz_axis));
      }
    }
    if (mask) atomicOr(&sh_mask, mask);
    __syncthreads();
    unsigned m = sh_mask;
    __syncthreads();
    if ((m & p.all_mask) == p.all_mask) {
      if (threadIdx.x == 0) atomicOr(&rb->viol_mask, m);
      break;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && sh_mask) atomicOr(&rb->viol_mask, sh_mask);
  // vals[0] = coeffs.first(); vals[1+v] = the candidate slope in[e_v] of axis v (:288-289)
  if (blockIdx.x == 0 && threadIdx.x == 0) rb->vals[0] = in[0];
  if (blockIdx.x == 0 && threadIdx.x < p.ndim)
    rb->vals[1 + threadIdx.x] = p.shape[threadIdx.x] >= 2 ? in[p.str[threadIdx.x]] : 0.0;
}
void launch_classify(Ctx& ctx, const double* in, const Shape& shape, Readback* rb_dev) {
  ClsParams p;
  memset(&p, 0, sizeof(p));
  p.ndim = (int)shape.size();
  GTP_CHECK(p.ndim <= MAXD, GTP_ERR_ARG, "ndim exceeds GTP_MAX_NDIM");
  p.total = prod(shape);
  for (int d = 0; d < p.ndim; d++) p.shape[d] = (unsigned)shape[d];
  {
    long long st = 1;
    for (int d = p.ndim - 1; d >= 0; --d) {
      p.str[d] = st;
      st *= (long long)shape[d];
    }
  }
  p.all_mask = p.ndim >= 32 ? 0xffffffffu : ((1u << p.ndim) - 1u);
  GTP_CUDA(cudaMemsetAsync(&rb_dev->viol_mask, 0, sizeof(unsigned), ctx.stream));
  int grid = (int)std::max<u64>(1, std::min<u64>((p.total + 255) / 256, (u64)ctx.sm_count * 4));
  GTP_LAUNCH(ctx, k_classify, grid, 256, 0, in, p, rb_dev);
}

__global__ void __launch_bounds__(256) k_classify_small(const double* __restrict__ in, const ClsParams p, Readback* rb,
                                                        unsigned long long seq) {
  __shared__ unsigned sh_mask;
  if (threadIdx.x == 0) sh_mask = 0;
  __syncthreads();
  unsigned mask = 0;
  for (u64 lin = threadIdx.x; lin < p.total; lin += blockDim.x) {
    double x = in[lin];
    if (x != 0.0) {
      u64 rem = lin;
      int nz_axis = -1, nz_count = 0;
      unsigned nz_val = 0;
      for (int d = p.ndim - 1; d >= 0; --d) {
        unsigned i = (unsigned)(rem % p.shape[d]);
        rem /= p.shape[d];
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
  if (mask) atomicOr(&sh_mask, mask);
  __syncthreads();
  if (threadIdx.x < p.ndim) rb->vals[1 + threadIdx.x] = p.shape[threadIdx.x] >= 2 ? in[p.str[threadIdx.x]] : 0.0;
  if (threadIdx.x == 0) {
    rb->vals[0] = in[0];
    rb->viol_mask = sh_mask;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) rb->seq = seq;   // published last
}

bool classify_small_zero_copy(Ctx& ctx, const double* in, const Shape& shape) {
  const u64 total = prod(shape);
  if (total > 8192 || !ctx.rb_host_dev || shape.size() > (size_t)MAXD) return false;
  ClsParams p;
  memset(&p, 0, sizeof(p));
  p.ndim = (int)shape.size();
  p.total = total;
  for (int d = 0; d < p.ndim; d++) p.shape[d] = (unsigned)shape[d];
  long long st = 1;
  for (int d = p.ndim - 1; d >= 0; --d) {
    p.str[d] = st;
    st *= (long long)shape[d];
  }
  p.all_mask = p.ndim >= 32 ? 0xffffffffu : ((1u << p.ndim) - 1u);
  const unsigned long long seq = ++ctx.rb_seq;
  GTP_LAUNCH(ctx, k_classify_small, 1, 256, 0, in, p, ctx.rb_host_dev, seq);
  // spin on the mapped page; fall back to a stream query now and then so a failed launch cannot hang the host
  for (unsigned long long spins = 0; ctx.rb_host->seq != seq; ++spins) {
    if ((spins & 0xfffff) == 0xfffff) {
      cudaError_t e = cudaStreamQuery(ctx.stream);
      if (e != cudaSuccess && e != cudaErrorNotReady) GTP_CUDA(e);
      if (e == cudaSuccess && ctx.rb_host->seq != seq) {   // stream drained but nothing published: treat as an error
        GTP_CUDA(cudaStreamSynchronize(ctx.stream));
        if (ctx.rb_host->seq != seq) throw Error(GTP_ERR_CUDA, "classification read-back was not published");
      }
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);   // the payload is read only after its sequence number
  return true;
}

__global__ void __launch_bounds__(256) k_eq(const double* __restrict__ a, const double* __restrict__ b, u64 n, Readback* rb) {
  u64 stride = (u64)gridDim.x * blockDim.x;
  bool ne = false;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) ne |= !(a[i] == b[i]);
  if (__syncthreads_or(ne) && threadIdx.x == 0) rb->flag = 0;
}
void launch_eq(Ctx& ctx, const double* a, const double* b, u64 n, Readback* rb_dev) {
  unsigned one = 1;
  GTP_CUDA(cudaMemcpyAsync(&rb_dev->flag, &one, sizeof(unsigned), cudaMemcpyHostToDevice, ctx.stream));
  int grid = (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)ctx.sm_count * 8));
  GTP_LAUNCH(ctx, k_eq, grid, 256, 0, a, b, n, rb_dev);
}

__global__ void k_gather_strided(const double* __restrict__ in, u64 stride, u64 len, u64 count, double* out) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = i < len ? in[i * stride] : 0.0;
}
void launch_gather_strided(Ctx& ctx, const double* in, u64 stride, u64 len, u64 count, double* out) {
  if (count == 0) return;
  GTP_LAUNCH(ctx, k_gather_strided, (unsigned)((count + 255) / 256), 256, 0, in, stride, len, count, out);
}

}  // namespace gtp
