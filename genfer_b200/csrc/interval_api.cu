// Interval<F64> TaylorPoly on the device (SURVEY 8 f3): the reference's --bounds number type (src/interval.rs: lo/hi pairs, every
// operation widened by one ulp on each side through integer bit operations, number/f64.rs:127-171) behind the same operator
// surface as gtp_* -- `gti_*`, one entry point per TaylorPoly method the host evaluator calls.  It exists so that north_star's
// check 2 ("results fall inside the reference's --bounds interval enclosure") runs at GPU speed on every program.
//
// The generic TaylorPoly<T> code of the reference (multivariate_taylor.rs) is what runs there with T = Interval<F64>; here the
// same dispatch (shape algebra, zero / one / constant fast paths of Mul and Div, result-shape rules of Div / exp / log) sits on
// the host and the arithmetic is done by generic kernels, one thread per output coefficient:
//   * element-wise / gather family and the truncated product visit their terms in the reference's order (so these agree with
//     the reference's interval results bit for bit: interval addition and multiplication are not associative once widened);
//   * div / exp / log are evaluated coefficient-wise over total-degree wavefronts (the recurrences of kernels_wave.cu written
//     per coefficient).  Their widening sequence differs from the reference's slice-wise recursion: the result is a valid
//     enclosure of the same quantity, a few ulps wider or narrower than the reference's.
// Mul's linear fast path (:1052-1061) and subst_var's geometric-scaling path (:555-568) are not special-cased: the general
// product / Horner loop enclose the same polynomial with the same stored shape.  PARITY UNPINNED, like the oracle's interval
// instantiation: no reference fixture runs with --bounds.
#include <cmath>

#include "interval.cuh"
#include "kernels.cuh"

using namespace gtp;
using gti::Iv;

struct gti_poly {
  BufP buf;           // 2 * len doubles: (lo, hi) pairs, row-major over `shape`
  u64 off = 0;        // in intervals
  Shape shape, degrees;
  bool known = false;   // `first` (coefficient 0) is known on the host
  Iv first{0.0, 0.0};
  const Iv* ptr() const { return reinterpret_cast<const Iv*>(buf->d) + off; }
  Iv* mptr() { return reinterpret_cast<Iv*>(buf->d) + off; }
  u64 len() const { return prod(shape); }
};
using IvP = std::unique_ptr<gti_poly>;

namespace {

constexpr int IVD = GTP_MAX_NDIM;
// Non-unit axes a product / recurrence kernel handles: the kernels keep their per-axis state in arrays of E entries; tensors
// of up to IVE non-unit axes run on the E = IVE instantiation, wider ones on E = IVD (more local memory per thread).
constexpr int IVE = 12;

// ------------------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------------------
struct IvEwP {
  int ndim, op, fax, s_by_val;
  u64 total;
  unsigned ext[IVD], a_ext[IVD], b_ext[IVD];
  long long a_str[IVD], b_str[IVD], o_str[IVD];
  long long a_base, b_base, o_base;
  const Iv* a;
  const Iv* b;
  Iv* out;
  const Iv* fac;
  const unsigned char* keep;
  const Iv* s;
  Iv s_val;
};
__global__ void __launch_bounds__(256) k_iv_ew(const IvEwP p) {
  const u64 stride = (u64)gridDim.x * blockDim.x;
  const Iv zero = gti::iv(0.0, 0.0);
  for (u64 lin = (u64)blockIdx.x * blockDim.x + threadIdx.x; lin < p.total; lin += stride) {
    u64 rem = lin;
    long long ao = p.a_base, bo = p.b_base, oo = p.o_base;
    bool a_ok = true, b_ok = true;
    unsigned fidx = 0;
    for (int d = p.ndim - 1; d >= 0; --d) {
      const unsigned e = p.ext[d];
      const unsigned i = (unsigned)(rem % e);
      rem /= e;
      ao += (long long)i * p.a_str[d];
      bo += (long long)i * p.b_str[d];
      oo += (long long)i * p.o_str[d];
      a_ok &= i < p.a_ext[d];
      b_ok &= i < p.b_ext[d];
      if (d == p.fax) fidx = i;
    }
    const bool first = lin == 0;
    Iv sv = zero;
    if (p.op == EW_SCALE_DEV || p.op == EW_DIV_DEV || p.op == EW_ADD_FIRST || p.op == EW_SUB_FIRST || p.op == EW_RSUB_FIRST)
      sv = p.s_by_val ? p.s_val : p.s[0];
    Iv r;
    switch (p.op) {
      case EW_COPY: r = p.fac ? gti::iv_mul(p.a[ao], p.fac[fidx]) : p.a[ao]; break;   // `*x *= factor`
      case EW_ADD: case EW_SUB:
        r = zero;
        if (a_ok) r = gti::iv_add(r, p.a[ao]);
        if (b_ok) r = p.op == EW_ADD ? gti::iv_add(r, p.b[bo]) : gti::iv_sub(r, p.b[bo]);
        break;
      case EW_MASK: r = p.keep[fidx] ? p.a[ao] : zero; break;
      case EW_SCALE_DEV: r = gti::iv_mul(sv, p.a[ao]); break;
      case EW_DIV_DEV: r = gti::iv_div(p.a[ao], sv); break;
      case EW_NEG: r = gti::iv_neg(p.a[ao]); break;
      case EW_ADD_FIRST: r = first ? gti::iv_add(p.a[ao], sv) : p.a[ao]; break;
      case EW_SUB_FIRST: r = first ? gti::iv_sub(p.a[ao], sv) : p.a[ao]; break;
      default: r = gti::iv_neg(first ? gti::iv_sub(p.a[ao], sv) : p.a[ao]); break;   // EW_RSUB_FIRST
    }
    p.out[oo] = r;
  }
}

// general truncated product in the reference's nesting order (`mul` :984-1012): see k_mul_ordered
template <int E>
struct IvMulP {
  int ne;
  unsigned xs[E], ys[E], rs[E];
  long long xstr[E], ystr[E];
  u64 total;
  const Iv* x;
  const Iv* y;
  Iv* out;
};
template <int E>
__global__ void __launch_bounds__(128) k_iv_mul(const IvMulP<E> p) {
  const u64 gstride = (u64)gridDim.x * blockDim.x;
  const int NE = p.ne;
  for (u64 lin = (u64)blockIdx.x * blockDim.x + threadIdx.x; lin < p.total; lin += gstride) {
    unsigned k[E], lo[E], hi[E], j[E];
    u64 rem = lin;
    bool empty = false;
    for (int d = NE - 1; d >= 0; --d) {
      k[d] = (unsigned)(rem % p.rs[d]);
      rem /= p.rs[d];
      lo[d] = (k[d] + 1 > p.ys[d]) ? k[d] + 1 - p.ys[d] : 0;
      hi[d] = (k[d] + 1 < p.xs[d]) ? k[d] + 1 : p.xs[d];
      empty |= hi[d] <= lo[d];
    }
    Iv total = gti::iv(0.0, 0.0);
    if (!empty) {
      long long xo = 0, yo = 0;
      for (int d = 0; d < NE - 1; d++) {
        j[d] = lo[d];
        xo += (long long)lo[d] * p.xstr[d];
        yo += (long long)(k[d] - lo[d]) * p.ystr[d];
      }
      const long long xsl = p.xstr[NE - 1], ysl = p.ystr[NE - 1];
      const unsigned kl = k[NE - 1], lol = lo[NE - 1], hil = hi[NE - 1];
      while (true) {
        Iv inner = gti::iv(0.0, 0.0);   // mul_1d: from zero, then `*z += o`
        const Iv* xp = p.x + xo + (long long)lol * xsl;
        const Iv* yp = p.y + yo + (long long)(kl - lol) * ysl;
        for (unsigned jl = lol; jl < hil; jl++) {
          inner = gti::iv_add(inner, gti::iv_mul(*xp, *yp));
          xp += xsl;
          yp -= ysl;
        }
        total = gti::iv_add(total, inner);
        bool advanced = false;
        for (int dd = NE - 2; dd >= 0 && !advanced; --dd) {
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
        if (!advanced) break;
      }
    }
    p.out[lin] = total;
  }
}

// div / exp / log, one total-degree level per launch: every coefficient of the level is an explicit function of coefficients of
// lower levels (the forward substitutions of kernels_wave.cu, per coefficient).  op 0: r = x / y;  1: exp(x);  2: log(x).
template <int E>
struct IvLevP {
  int op, ne;
  unsigned rs[E], xs[E], ys[E];
  long long rstr[E], xstr[E], ystr[E];
  u64 outer_total;   // prod(rs[0 .. ne-2])
  const Iv* x;
  const Iv* y;
  Iv* r;
  Iv* q;             // log: unscaled quotients
  int has_seed;
  Iv seed;           // exp / log of the constant term from the host's libm when the host knows it
};
template <int E>
__device__ __forceinline__ void iv_level_body(const IvLevP<E>& p, unsigned level, u64 first, u64 gstride) {
  const int ne = p.ne;
  const Iv zero = gti::iv(0.0, 0.0);
  for (u64 lin = first; lin < p.outer_total; lin += gstride) {
    unsigned k[E];
    u64 rem = lin;
    unsigned sum = 0;
    for (int d = ne - 2; d >= 0; --d) {
      k[d] = (unsigned)(rem % p.rs[d]);
      rem /= p.rs[d];
      sum += k[d];
    }
    if (sum > level) continue;
    k[ne - 1] = level - sum;
    if (k[ne - 1] >= p.rs[ne - 1]) continue;
    long long ro = 0, xo = 0;
    bool in_x = true;
    int a = -1;
    for (int d = 0; d < ne; d++) {
      ro += (long long)k[d] * p.rstr[d];
      xo += (long long)k[d] * p.xstr[d];
      in_x &= k[d] < p.xs[d];
      if (a < 0 && k[d] != 0) a = d;
    }
    if (a < 0) {   // the constant term
      if (p.op == 0) p.r[0] = gti::iv_div(p.x[0], p.y[0]);
      else p.r[0] = p.has_seed ? p.seed : (p.op == 1 ? gti::iv_exp(p.x[0]) : gti::iv_log(p.x[0]));
      continue;
    }
    unsigned lo[E], hi[E], m[E];   // inclusive bounds of the summation index
    if (p.op == 0) {
      // r[k] = ((-sum_{m <= k, m != k, k - m < ys} r[m] * y[k - m]) + x[k]) / y[0]          (:1170-1191)
      bool any = true;
      for (int d = 0; d < ne; d++) {
        lo[d] = k[d] + 1 > p.ys[d] ? k[d] + 1 - p.ys[d] : 0;
        hi[d] = k[d];
        m[d] = lo[d];
      }
      Iv s = zero;
      while (any) {
        bool is_k = true;
        long long mo = 0, yo = 0;
        for (int d = 0; d < ne; d++) {
          is_k &= m[d] == k[d];
          mo += (long long)m[d] * p.rstr[d];
          yo += (long long)(k[d] - m[d]) * p.ystr[d];
        }
        if (!is_k) s = gti::iv_add(s, gti::iv_mul(p.r[mo], p.y[yo]));
        int d = ne - 1;
        for (; d >= 0; --d) {
          if (m[d] < hi[d]) { m[d]++; break; }
          m[d] = lo[d];
        }
        any = d >= 0;
      }
      Iv num = gti::iv_neg(s);
      if (in_x) num = gti::iv_add(num, p.x[xo]);
      p.r[ro] = gti::iv_div(num, p.y[0]);
    } else if (p.op == 1) {
      // r[k] = (sum_{j: j_i = 0 (i < a), 1 <= j_a <= k_a, j_b <= k_b (b > a)} (x[j] * j_a) * r[k - j]) / k_a    (:1302-1316)
      bool any = true;
      for (int d = 0; d < ne; d++) {
        if (d < a) { lo[d] = 0; hi[d] = 0; }
        else if (d == a) { lo[d] = 1; hi[d] = min(k[d], p.xs[d] - 1); }
        else { lo[d] = 0; hi[d] = min(k[d], p.xs[d] - 1); }
        m[d] = lo[d];
        any = any && hi[d] >= lo[d];
      }
      Iv s = zero;
      while (any) {
        long long jo = 0, mo = 0;
        for (int d = 0; d < ne; d++) {
          jo += (long long)m[d] * p.xstr[d];
          mo += (long long)(k[d] - m[d]) * p.rstr[d];
        }
        s = gti::iv_add(s, gti::iv_mul(gti::iv_mul(p.x[jo], gti::iv_from_u32(m[a])), p.r[mo]));
        int d = ne - 1;
        for (; d >= 0; --d) {
          if (m[d] < hi[d]) { m[d]++; break; }
          m[d] = lo[d];
        }
        any = d >= 0;
      }
      p.r[ro] = gti::iv_div(s, gti::iv_from_u32(k[a]));
    } else {
      // log (:1355-1385): q[k] = ((-T2) + ((-T1) + k_a x[k])) / x[0],  r[k] = q[k] / k_a
      Iv t1 = zero, t2 = zero;
      {   // T1 = sum_{m_i = 0 (i < a), max(1, k_a - xs_a + 1) <= m_a <= k_a - 1, m_b <= k_b, k_b - m_b < xs_b} x[k - m] * (r[m] * m_a)
        bool any = k[a] >= 2;
        for (int d = 0; d < ne; d++) {
          if (d < a) { lo[d] = 0; hi[d] = 0; }
          else if (d == a) { lo[d] = max(1u, k[d] + 1 > p.xs[d] ? k[d] + 1 - p.xs[d] : 0u); hi[d] = k[d] - 1; }
          else { lo[d] = k[d] + 1 > p.xs[d] ? k[d] + 1 - p.xs[d] : 0; hi[d] = k[d]; }
          m[d] = lo[d];
          any = any && hi[d] >= lo[d];
        }
        while (any) {
          long long mo = 0, jo = 0;
          for (int d = 0; d < ne; d++) {
            mo += (long long)m[d] * p.rstr[d];
            jo += (long long)(k[d] - m[d]) * p.xstr[d];
          }
          t1 = gti::iv_add(t1, gti::iv_mul(p.x[jo], gti::iv_mul(p.r[mo], gti::iv_from_u32(m[a]))));
          int d = ne - 1;
          for (; d >= 0; --d) {
            if (m[d] < hi[d]) { m[d]++; break; }
            m[d] = lo[d];
          }
          any = d >= 0;
        }
      }
      {   // T2 = sum_{m_i = k_i (i <= a), m_b <= k_b, k_b - m_b < xs_b (b > a), m != k} q[m] * x[0 .., k_b - m_b]
        bool any = true;
        for (int d = 0; d < ne; d++) {
          if (d <= a) { lo[d] = k[d]; hi[d] = k[d]; }
          else { lo[d] = k[d] + 1 > p.xs[d] ? k[d] + 1 - p.xs[d] : 0; hi[d] = k[d]; }
          m[d] = lo[d];
        }
        while (any) {
          bool is_k = true;
          long long mo = 0, jo = 0;
          for (int d = 0; d < ne; d++) {
            is_k &= m[d] == k[d];
            mo += (long long)m[d] * p.rstr[d];
            if (d > a) jo += (long long)(k[d] - m[d]) * p.xstr[d];
          }
          if (!is_k) t2 = gti::iv_add(t2, gti::iv_mul(p.q[mo], p.x[jo]));
          int d = ne - 1;
          for (; d >= 0; --d) {
            if (m[d] < hi[d]) { m[d]++; break; }
            m[d] = lo[d];
          }
          any = d >= 0;
        }
      }
      Iv num = gti::iv_neg(t1);
      if (in_x) num = gti::iv_add(num, gti::iv_mul(gti::iv_from_u32(k[a]), p.x[xo]));
      num = gti::iv_add(gti::iv_neg(t2), num);
      const Iv qv = gti::iv_div(num, p.x[0]);
      p.q[ro] = qv;
      p.r[ro] = gti::iv_div(qv, gti::iv_from_u32(k[a]));
    }
  }
}

template <int E>
__global__ void __launch_bounds__(128) k_iv_level(const IvLevP<E> p, unsigned level) {
  iv_level_body(p, level, (u64)blockIdx.x * blockDim.x + threadIdx.x, (u64)gridDim.x * blockDim.x);
}
// Small tensors (1-d and thin 2-d series: hundreds of levels of a handful of coefficients each): ALL levels in one single-CTA
// launch, a block barrier between levels (the level's coefficients are written and read by this CTA only).
template <int E>
__global__ void __launch_bounds__(256) k_iv_levels_cta(const IvLevP<E> p, unsigned levels) {
  for (unsigned level = 0; level < levels; level++) {
    iv_level_body(p, level, threadIdx.x, blockDim.x);
    __syncthreads();
  }
}

// shift_down (:514-536) on the (outer, len, inner) view of the axis: slot 0 = in[n] + (in[0] + .. + in[n-1]), the rest moves down
__global__ void __launch_bounds__(256) k_iv_shift_down(const Iv* in, Iv* out, u64 outer, u64 len, u64 inner, u64 n, u64 out_len) {
  const u64 total = outer * out_len * inner, stride = (u64)gridDim.x * blockDim.x;
  for (u64 lin = (u64)blockIdx.x * blockDim.x + threadIdx.x; lin < total; lin += stride) {
    const u64 i = lin % inner, j = (lin / inner) % out_len, o = lin / (inner * out_len);
    const Iv* src = in + o * len * inner + i;
    Iv v;
    if (len <= n + 1) {        // sum_axis over the whole axis
      v = gti::iv(0.0, 0.0);
      for (u64 t = 0; t < len; t++) v = gti::iv_add(v, src[t * inner]);
    } else if (j == 0) {       // result[0] = in[n] + sum_{t < n} in[t]
      Iv s = gti::iv(0.0, 0.0);
      for (u64 t = 0; t < n; t++) s = gti::iv_add(s, src[t * inner]);
      v = gti::iv_add(src[n * inner], s);
    } else {
      v = src[(n + j) * inner];
    }
    out[lin] = v;
  }
}
__global__ void k_iv_gather(const Iv* in, u64 stride, u64 len, u64 count, Iv* out) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = i < len ? in[i * stride] : gti::iv(0.0, 0.0);
}

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
IvP mk(BufP buf, u64 off, Shape shape, Shape degrees) {
  GTP_CHECK(shape.size() == degrees.size(), GTP_ERR_SHAPE, "coeffs.ndim() != degrees_p1.len()");
  GTP_CHECK(shape.size() <= (size_t)GTP_MAX_NDIM, GTP_ERR_ARG, "ndim exceeds GTP_MAX_NDIM");
  for (size_t i = 0; i < shape.size(); i++) GTP_CHECK(0 < shape[i] && shape[i] <= degrees[i], GTP_ERR_SHAPE, "need 0 < shape[i] <= degrees_p1[i]");
  IvP p(new gti_poly());
  p->buf = std::move(buf);
  p->off = off;
  p->shape = std::move(shape);
  p->degrees = std::move(degrees);
  return p;
}
IvP fresh(Ctx& c, const Shape& shape, const Shape& degrees) { return mk(c.alloc(2 * std::max<u64>(prod(shape), 1)), 0, shape, degrees); }
IvP share(const gti_poly& a) { return IvP(new gti_poly(a)); }
IvP scalar(Ctx& c, Iv x, const Shape& degrees) {
  IvP p = fresh(c, Shape(degrees.size(), 1), degrees);
  GTP_CUDA(cudaMemcpyAsync(p->buf->d, &x, sizeof(Iv), cudaMemcpyHostToDevice, c.stream));   // pageable source: staged before return
  p->known = true;
  p->first = x;
  return p;
}
Iv first_of(Ctx& c, const gti_poly& p) {
  if (p.known) return p.first;
  Iv v;
  GTP_CUDA(cudaMemcpyAsync(&v, p.ptr(), sizeof(Iv), cudaMemcpyDeviceToHost, c.stream));
  c.sync();
  gti_poly& m = const_cast<gti_poly&>(p);   // cache of an immutable value
  m.known = true;
  m.first = v;
  return v;
}
bool is_zero(Ctx& c, const gti_poly& p) { return p.len() == 1 && gti::iv_is_zero(first_of(c, p)); }
bool is_one(Ctx& c, const gti_poly& p) { return p.len() == 1 && gti::iv_is_one(first_of(c, p)); }

Shape min_degrees(const gti_poly& a, const gti_poly& b) {   // :114-127
  Shape d(std::max(a.degrees.size(), b.degrees.size()), UNB);
  for (size_t v = 0; v < d.size(); v++) {
    if (v < a.degrees.size()) d[v] = std::min(d[v], a.degrees[v]);
    if (v < b.degrees.size()) d[v] = std::min(d[v], b.degrees[v]);
  }
  return d;
}
Shape max_shape(const gti_poly& a, const gti_poly& b) {   // :129-148
  Shape s(std::max(a.shape.size(), b.shape.size()), 1);
  for (size_t v = 0; v < s.size(); v++) {
    if (v < a.shape.size()) s[v] = std::max(s[v], a.shape[v]);
    if (v < b.shape.size()) s[v] = std::max(s[v], b.shape[v]);
    if (v < a.degrees.size()) s[v] = std::min(s[v], a.degrees[v]);
    if (v < b.degrees.size()) s[v] = std::min(s[v], b.degrees[v]);
  }
  return s;
}
Shape sum_shape(const gti_poly& a, const gti_poly& b) {   // :150-170
  Shape s(std::max(a.shape.size(), b.shape.size()), 0);
  for (size_t v = 0; v < s.size(); v++) {
    if (v < a.shape.size()) s[v] += a.shape[v] - 1;
    if (v < b.shape.size()) s[v] += b.shape[v] - 1;
    s[v] += 1;
    if (v < a.degrees.size()) s[v] = std::min(s[v], a.degrees[v]);
    if (v < b.degrees.size()) s[v] = std::min(s[v], b.degrees[v]);
  }
  return s;
}
void broadcast(gti_poly& x, gti_poly& y) {   // :832-852
  if (x.degrees.size() < y.degrees.size()) x.degrees.insert(x.degrees.end(), y.degrees.begin() + x.degrees.size(), y.degrees.end());
  else if (y.degrees.size() < x.degrees.size()) y.degrees.insert(y.degrees.end(), x.degrees.begin() + y.degrees.size(), x.degrees.end());
  if (x.shape.size() < y.shape.size()) x.shape.resize(y.shape.size(), 1);
  if (y.shape.size() < x.shape.size()) y.shape.resize(x.shape.size(), 1);
}
Shape strides_of(const Shape& shape) {
  Shape st(shape.size(), 1);
  for (int i = (int)shape.size() - 2; i >= 0; --i) st[i] = st[i + 1] * shape[i + 1];
  return st;
}

struct Opnd {
  const Iv* p = nullptr;
  Shape shape, lo, valid;
};
void ew(Ctx& c, int op, const Shape& box, const Opnd& a, const Opnd* b, Iv* out, const Shape& out_shape, const Shape& out_lo, int fax = -1,
        const Iv* fac = nullptr, const unsigned char* keep = nullptr, const Iv* s_dev = nullptr, const Iv* s_host = nullptr) {
  const int nd = (int)box.size();
  const u64 total = prod(box);
  if (total == 0) return;
  IvEwP p;
  memset(&p, 0, sizeof(p));
  Shape ast = strides_of(a.shape), ost = strides_of(out_shape), bst;
  if (b) bst = strides_of(b->shape);
  int n = 0;
  p.fax = -1;
  for (int d = 0; d < nd; d++) {
    p.a_base += (long long)(a.lo.empty() ? 0 : a.lo[d]) * (long long)ast[d];
    if (b) p.b_base += (long long)(b->lo.empty() ? 0 : b->lo[d]) * (long long)bst[d];
    p.o_base += (long long)(out_lo.empty() ? 0 : out_lo[d]) * (long long)ost[d];
    if (box[d] == 1 && d != fax) continue;   // unit axes carry no index
    p.ext[n] = (unsigned)box[d];
    p.a_ext[n] = (unsigned)(a.valid.empty() ? box[d] : std::min<u64>(a.valid[d], box[d]));
    p.b_ext[n] = (unsigned)((b && !b->valid.empty()) ? std::min<u64>(b->valid[d], box[d]) : box[d]);
    p.a_str[n] = (long long)ast[d];
    p.b_str[n] = b ? (long long)bst[d] : 0;
    p.o_str[n] = (long long)ost[d];
    if (d == fax) p.fax = n;
    n++;
  }
  p.ndim = n;
  p.op = op;
  p.total = total;
  p.a = a.p;
  p.b = b ? b->p : nullptr;
  p.out = out;
  p.fac = fac;
  p.keep = keep;
  p.s = s_dev;
  p.s_by_val = s_host ? 1 : 0;
  if (s_host) p.s_val = *s_host;
  const int grid = (int)std::max<u64>(1, std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16));
  GTP_LAUNCH(c, k_iv_ew, grid, 256, 0, p);
}

IvP copy_box(Ctx& c, const gti_poly& a, const Shape& lo, const Shape& ext, const Shape& degrees) {
  IvP r = fresh(c, ext, degrees);
  Opnd A;
  A.p = a.ptr();
  A.shape = a.shape;
  A.lo = lo;
  ew(c, EW_COPY, ext, A, nullptr, r->mptr(), ext, {});
  return r;
}
IvP truncate_degrees(Ctx& c, const gti_poly& a, const Shape& d) {   // :195-204
  Shape nd = a.degrees, ns = a.shape;
  bool cut = false, cut_inner = false;
  for (size_t v = 0; v < a.degrees.size(); v++) {
    nd[v] = std::min(a.degrees[v], d[v]);
    if (a.shape[v] > d[v]) {
      ns[v] = d[v];
      cut = true;
      if (v > 0) cut_inner = true;
    }
  }
  if (!cut) {
    IvP r = share(a);
    r->degrees = nd;
    return r;
  }
  if (!cut_inner) {
    IvP r = mk(a.buf, a.off, ns, nd);   // prefix of the same buffer
    r->known = a.known;
    r->first = a.first;
    return r;
  }
  return copy_box(c, a, Shape(ns.size(), 0), ns, nd);
}
IvP ew_scalar(Ctx& c, int op, const gti_poly& a, const gti_poly& sp, const Shape& degrees) {
  IvP r = fresh(c, a.shape, degrees);
  Opnd A;
  A.p = a.ptr();
  A.shape = a.shape;
  ew(c, op, a.shape, A, nullptr, r->mptr(), a.shape, {}, -1, nullptr, nullptr, sp.known ? nullptr : sp.ptr(), sp.known ? &sp.first : nullptr);
  return r;
}

IvP poly_add(Ctx& c, const gti_poly& a0, const gti_poly& b0, bool subtract) {   // :854-937
  Shape rd = min_degrees(a0, b0);
  gti_poly a = a0, b = b0;
  broadcast(a, b);
  IvP at = truncate_degrees(c, a, rd), bt = truncate_degrees(c, b, rd);
  if (bt->len() == 1) return ew_scalar(c, subtract ? EW_SUB_FIRST : EW_ADD_FIRST, *at, *bt, rd);
  if (at->len() == 1) return ew_scalar(c, subtract ? EW_RSUB_FIRST : EW_ADD_FIRST, *bt, *at, rd);
  Shape shape = max_shape(*at, *bt);
  IvP r = fresh(c, shape, rd);
  Opnd A, B;
  A.p = at->ptr(); A.shape = at->shape; A.valid = at->shape;
  B.p = bt->ptr(); B.shape = bt->shape; B.valid = bt->shape;
  ew(c, subtract ? EW_SUB : EW_ADD, shape, A, &B, r->mptr(), shape, {});
  return r;
}
IvP poly_neg(Ctx& c, const gti_poly& a) {
  IvP r = fresh(c, a.shape, a.degrees);
  Opnd A;
  A.p = a.ptr();
  A.shape = a.shape;
  ew(c, EW_NEG, a.shape, A, nullptr, r->mptr(), a.shape, {});
  return r;
}

template <int E>
void launch_iv_mul_e(Ctx& c, const Iv* x, const Shape& xs, const Iv* y, const Shape& ys, Iv* out, const Shape& rs) {
  const int nd = (int)rs.size();
  IvMulP<E> p;
  memset(&p, 0, sizeof(p));
  Shape xst = strides_of(xs), yst = strides_of(ys);
  int ne = 0;
  for (int d = 0; d < nd; d++) {
    if (rs[d] == 1) continue;   // unit result axis: only index 0 of both operands contributes
    p.xs[ne] = (unsigned)xs[d]; p.ys[ne] = (unsigned)ys[d]; p.rs[ne] = (unsigned)rs[d];
    p.xstr[ne] = (long long)xst[d]; p.ystr[ne] = (long long)yst[d];
    ne++;
  }
  if (ne == 0) {
    p.xs[0] = p.ys[0] = p.rs[0] = 1;
    p.xstr[0] = p.ystr[0] = 1;
    ne = 1;
  }
  p.ne = ne;
  p.total = prod(rs);
  p.x = x; p.y = y; p.out = out;
  if (p.total == 0) return;
  const int grid = (int)std::max<u64>(1, std::min<u64>((p.total + 127) / 128, (u64)c.sm_count * 64));
  GTP_LAUNCH(c, k_iv_mul<E>, grid, 128, 0, p);
}
int nonunit_axes(const Shape& s) { return (int)std::count_if(s.begin(), s.end(), [](u64 x) { return x != 1; }); }
void launch_iv_mul(Ctx& c, const Iv* x, const Shape& xs, const Iv* y, const Shape& ys, Iv* out, const Shape& rs) {
  if (nonunit_axes(rs) <= IVE) launch_iv_mul_e<IVE>(c, x, xs, y, ys, out, rs);
  else launch_iv_mul_e<IVD>(c, x, xs, y, ys, out, rs);
}

IvP poly_mul(Ctx& c, const gti_poly& a0, const gti_poly& b0) {   // :1014-1072
  Shape d = min_degrees(a0, b0);
  if (is_zero(c, a0) || is_zero(c, b0)) return scalar(c, gti::iv(0.0, 0.0), d);
  gti_poly a = a0, b = b0;
  broadcast(a, b);
  Shape shape = sum_shape(a, b);
  IvP at = truncate_degrees(c, a, d), bt = truncate_degrees(c, b, d);
  auto with_deg = [&](IvP p) { p->degrees = d; return p; };
  if (is_one(c, *at)) return with_deg(share(*bt));
  if (is_one(c, *bt)) return with_deg(share(*at));
  if (at->len() == 1) return ew_scalar(c, EW_SCALE_DEV, *bt, *at, d);
  if (bt->len() == 1) return ew_scalar(c, EW_SCALE_DEV, *at, *bt, d);
  IvP r = fresh(c, shape, d);
  launch_iv_mul(c, at->ptr(), at->shape, bt->ptr(), bt->shape, r->mptr(), shape);
  return r;
}

// div / exp / log by total-degree levels.  x, (y), r share ndim; r is dense over rs.
template <int E>
void run_levels_e(Ctx& c, int op, const gti_poly& x, const gti_poly* y, gti_poly& r, const Iv* seed) {
  const int nd = (int)r.shape.size();
  IvLevP<E> p;
  memset(&p, 0, sizeof(p));
  Shape xst = strides_of(x.shape), rst = strides_of(r.shape), yst;
  if (y) yst = strides_of(y->shape);
  int ne = 0;
  u64 levels = 1;
  for (int d = 0; d < nd; d++) {
    if (r.shape[d] == 1) continue;
    p.rs[ne] = (unsigned)r.shape[d]; p.xs[ne] = (unsigned)x.shape[d]; p.ys[ne] = y ? (unsigned)y->shape[d] : 1u;
    p.rstr[ne] = (long long)rst[d]; p.xstr[ne] = (long long)xst[d]; p.ystr[ne] = y ? (long long)yst[d] : 0;
    levels += r.shape[d] - 1;
    ne++;
  }
  if (ne == 0) {
    p.rs[0] = p.xs[0] = p.ys[0] = 1;
    ne = 1;
  }
  p.op = op;
  p.ne = ne;
  p.outer_total = 1;
  for (int d = 0; d < ne - 1; d++) p.outer_total *= p.rs[d];
  p.x = x.ptr();
  p.y = y ? y->ptr() : nullptr;
  p.r = r.mptr();
  BufP q;
  if (op == 2) {
    q = c.alloc(2 * std::max<u64>(prod(r.shape), 1));
    p.q = reinterpret_cast<Iv*>(q->d);
  }
  p.has_seed = seed ? 1 : 0;
  if (seed) p.seed = *seed;
  if (p.outer_total <= 2048 && levels <= (1u << 20)) {
    GTP_LAUNCH(c, k_iv_levels_cta<E>, 1, 256, 0, p, (unsigned)levels);
    return;
  }
  const int grid = (int)std::max<u64>(1, std::min<u64>((p.outer_total + 127) / 128, (u64)c.sm_count * 32));
  for (u64 t = 0; t < levels; t++) GTP_LAUNCH(c, k_iv_level<E>, grid, 128, 0, p, (unsigned)t);
}
void run_levels(Ctx& c, int op, const gti_poly& x, const gti_poly* y, gti_poly& r, const Iv* seed) {
  if (nonunit_axes(r.shape) <= IVE) run_levels_e<IVE>(c, op, x, y, r, seed);
  else run_levels_e<IVD>(c, op, x, y, r, seed);
}

IvP poly_div(Ctx& c, const gti_poly& a0, const gti_poly& b0) {   // :1194-1231
  gti_poly a = a0, b = b0;
  broadcast(a, b);
  Shape d = min_degrees(a, b);
  IvP at = truncate_degrees(c, a, d), bt = truncate_degrees(c, b, d);
  if (is_one(c, *bt)) { IvP r = share(*at); r->degrees = d; return r; }
  if (bt->len() == 1) return ew_scalar(c, EW_DIV_DEV, *at, *bt, d);
  Shape rs = d;
  for (size_t i = 0; i < rs.size(); i++)
    if (bt->shape[i] == 1) rs[i] = at->shape[i];
  for (u64 x : rs) GTP_CHECK(x != UNB, GTP_ERR_SHAPE, "division by a non-constant series needs bounded degrees");
  IvP r = fresh(c, rs, d);
  run_levels(c, 0, *at, bt.get(), *r, nullptr);
  return r;
}
IvP poly_exp_log(Ctx& c, const gti_poly& a, bool is_log) {   // :406-430
  Shape rs = a.degrees;
  for (size_t i = 0; i < rs.size(); i++)
    if (a.shape[i] == 1) rs[i] = 1;
  for (u64 x : rs) GTP_CHECK(x != UNB, GTP_ERR_SHAPE, "exp/log of a non-constant series needs bounded degrees");
  IvP r = fresh(c, rs, a.degrees);
  Iv seed;
  const Iv* sp = nullptr;
  if (a.known) {   // the host's libm, like the reference (interval.rs:264-276)
    seed = is_log ? gti::iv_log(a.first) : gti::iv_exp(a.first);
    sp = &seed;
  }
  run_levels(c, is_log ? 2 : 1, a, nullptr, *r, sp);
  return r;
}
IvP poly_pow(Ctx& c, const gti_poly& a, uint32_t e) {   // :433-451
  if (e == 0) return scalar(c, gti::iv(1.0, 1.0), {});
  if (e == 1) return share(a);
  IvP res = scalar(c, gti::iv(1.0, 1.0), {});
  IvP base = share(a);
  while (e > 0) {
    if (e & 1) res = poly_mul(c, *res, *base);
    base = poly_mul(c, *base, *base);
    e >>= 1;
  }
  return res;
}

// slice n.. along v scaled by the derivative / coefficient-expansion factors, built on the host in the reference's incremental
// order with interval arithmetic (:472-479, :499-507)
IvP slice_scale(Ctx& c, const gti_poly& a, u64 v, u64 n, int kind) {
  GTP_CHECK(v < a.degrees.size() && n < a.degrees[v], GTP_ERR_INDEX, "variable / order out of range");
  if (v >= a.shape.size()) return n == 0 ? share(a) : scalar(c, gti::iv(0.0, 0.0), a.degrees);
  Shape d = a.degrees;
  d[v] = sat_sub(d[v], n);
  if (n >= a.shape[v]) return scalar(c, gti::iv(0.0, 0.0), d);
  Shape ext = a.shape, lo(a.shape.size(), 0);
  ext[v] = a.shape[v] - n;
  lo[v] = n;
  std::vector<Iv> fac(ext[v]);
  if (kind == 0) {
    Iv f = gti::iv(1.0, 1.0);
    for (u64 i = 1; i <= n; i++) f = gti::iv_mul(f, gti::iv_from_u32((uint32_t)i));
    for (u64 k = 0; k < ext[v]; k++) {
      fac[k] = f;
      f = gti::iv_mul(f, gti::iv_div(gti::iv_from_u32((uint32_t)(n + k + 1)), gti::iv_from_u32((uint32_t)(k + 1))));
    }
  } else {
    Iv f = gti::iv(1.0, 1.0);
    fac[0] = f;
    for (u64 k = 1; k < ext[v]; k++) {
      f = gti::iv_mul(f, gti::iv_div(gti::iv_from_u32((uint32_t)(n + k)), gti::iv_from_u32((uint32_t)k)));
      fac[k] = f;
    }
  }
  BufP fb = c.alloc(2 * ext[v]);
  GTP_CUDA(cudaMemcpyAsync(fb->d, fac.data(), ext[v] * sizeof(Iv), cudaMemcpyHostToDevice, c.stream));
  IvP r = fresh(c, ext, d);
  Opnd A;
  A.p = a.ptr();
  A.shape = a.shape;
  A.lo = lo;
  ew(c, EW_COPY, ext, A, nullptr, r->mptr(), ext, {}, (int)v, reinterpret_cast<const Iv*>(fb->d));
  return r;
}
IvP poly_shift_down(Ctx& c, const gti_poly& a, u64 v, u64 n) {
  GTP_CHECK(v < a.degrees.size() && n < a.degrees[v], GTP_ERR_INDEX, "shift_down: variable / order out of range");
  if (v >= a.shape.size()) return share(a);
  Shape d = a.degrees;
  d[v] = sat_sub(d[v], n);
  Shape rs = a.shape;
  rs[v] = (a.shape[v] <= n + 1) ? 1 : a.shape[v] - n;
  IvP r = fresh(c, rs, d);
  u64 outer = 1, inner = 1;
  for (size_t i = 0; i < v; i++) outer *= a.shape[i];
  for (size_t i = v + 1; i < a.shape.size(); i++) inner *= a.shape[i];
  const u64 total = prod(rs);
  const int grid = (int)std::max<u64>(1, std::min<u64>((total + 255) / 256, (u64)c.sm_count * 16));
  GTP_LAUNCH(c, k_iv_shift_down, grid, 256, 0, a.ptr(), r->mptr(), outer, a.shape[v], inner, n, rs[v]);
  return r;
}
IvP poly_subst_var(Ctx& c, const gti_poly& self, u64 v, const gti_poly& subst) {   // :540-580 (zero path and Horner)
  if (v >= self.shape.size()) return share(self);
  Shape d = min_degrees(self, subst);
  gti_poly cs = self;
  cs.shape.resize(std::max(cs.shape.size(), d.size()), 1);
  Shape ext(cs.shape.size()), lo(cs.shape.size(), 0);
  for (size_t a = 0; a < ext.size(); a++) ext[a] = std::min(cs.shape[a], d[a]);
  if (is_zero(c, subst)) {
    Shape e2 = cs.shape;
    e2[v] = 1;
    return copy_box(c, cs, lo, e2, d);
  }
  IvP res = scalar(c, gti::iv(0.0, 0.0), d);
  ext[v] = 1;
  for (u64 i = cs.shape[v]; i-- > 0;) {
    lo[v] = i;
    IvP slice = copy_box(c, cs, lo, ext, d);
    IvP pr = poly_mul(c, *res, subst);
    res = poly_add(c, *pr, *slice, false);
  }
  return res;
}

template <class F> int wrap(gtp_ctx* ctx, F&& f) {
  try {
    if (ctx) GTP_CUDA(cudaSetDevice(ctx->device));
    f();
    return GTP_OK;
  } catch (const gtp::Error& e) {
    if (ctx) ctx->err = e.what();
    return e.code;
  } catch (const std::exception& e) {
    if (ctx) ctx->err = e.what();
    return GTP_ERR_ARG;
  }
}
Shape to_shape(const uint64_t* p, int n) { return p ? Shape(p, p + n) : Shape(); }
IvP make_var(Ctx& c, u64 v, Iv x, u64 stored, bool one_coeff, Shape degrees) {
  Shape shape(degrees.size(), 1);
  shape[v] = stored;
  Iv vals[2] = {x, one_coeff ? gti::iv(1.0, 1.0) : gti::iv(0.0, 0.0)};
  IvP p = fresh(c, shape, degrees);
  GTP_CUDA(cudaMemcpyAsync(p->buf->d, vals, stored * sizeof(Iv), cudaMemcpyHostToDevice, c.stream));
  p->known = true;
  p->first = x;
  return p;
}

}  // namespace

extern "C" {

int gti_from_scalar(gtp_ctx* c, double lo, double hi, gti_poly** out) { return wrap(c, [&] { *out = scalar(*c, gti::iv(lo, hi), {}).release(); }); }
int gti_zero_with(gtp_ctx* c, int ndim, const uint64_t* degrees, gti_poly** out) {
  return wrap(c, [&] { *out = scalar(*c, gti::iv(0.0, 0.0), to_shape(degrees, ndim)).release(); });
}
int gti_var(gtp_ctx* c, uint64_t v, double lo, double hi, uint64_t len, gti_poly** out) {   // :239-248
  return wrap(c, [&] {
    GTP_CHECK(v < (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "variable index too large");
    *out = make_var(*c, v, gti::iv(lo, hi), std::min<u64>(len, 2), len > 1, Shape(v + 1, len)).release();
  });
}
int gti_var_at_zero(gtp_ctx* c, uint64_t v, uint64_t len, gti_poly** out) {   // :228-237
  return wrap(c, [&] {
    GTP_CHECK(v < (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "variable index too large");
    *out = make_var(*c, v, gti::iv(0.0, 0.0), 2, len > 1, Shape(v + 1, len)).release();
  });
}
int gti_var_with_degrees_p1(gtp_ctx* c, uint64_t v, double lo, double hi, int ndim, const uint64_t* degrees, gti_poly** out) {   // :250-259
  return wrap(c, [&] {
    GTP_CHECK((int)v < ndim, GTP_ERR_INDEX, "variable index out of range");
    *out = make_var(*c, v, gti::iv(lo, hi), 2, degrees[v] > 1, to_shape(degrees, ndim)).release();
  });
}
// `data`: prod(shape) (lo, hi) pairs (pairs != 0) or prod(shape) doubles taken as point intervals (pairs == 0)
int gti_from_host(gtp_ctx* c, int ndim, const uint64_t* shape, const uint64_t* degrees, const double* data, int pairs, gti_poly** out) {
  return wrap(c, [&] {
    GTP_CHECK(out && data && ndim >= 0 && ndim <= GTP_MAX_NDIM, GTP_ERR_ARG, "bad arguments");
    IvP p = fresh(*c, to_shape(shape, ndim), to_shape(degrees, ndim));
    const u64 n = p->len();
    if (pairs) {
      GTP_CUDA(cudaMemcpyAsync(p->buf->d, data, n * sizeof(Iv), cudaMemcpyHostToDevice, c->stream));
    } else {
      std::vector<Iv> tmp(n);
      for (u64 i = 0; i < n; i++) tmp[i] = gti::iv_point(data[i]);
      GTP_CUDA(cudaMemcpyAsync(p->buf->d, tmp.data(), n * sizeof(Iv), cudaMemcpyHostToDevice, c->stream));
    }
    c->sync();
    *out = p.release();
  });
}
int gti_to_host(gtp_ctx* c, const gti_poly* p, double* out_pairs) {
  return wrap(c, [&] {
    GTP_CUDA(cudaMemcpyAsync(out_pairs, p->ptr(), p->len() * sizeof(Iv), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
  });
}
void gti_free(gtp_ctx* c, gti_poly* p) {
  if (c) cudaSetDevice(c->device);
  delete p;
}
int gti_ndim(const gti_poly* p) { return (int)p->shape.size(); }
uint64_t gti_len(const gti_poly* p) { return p->len(); }
void gti_shape(const gti_poly* p, uint64_t* out) { std::copy(p->shape.begin(), p->shape.end(), out); }
void gti_degrees_p1(const gti_poly* p, uint64_t* out) { std::copy(p->degrees.begin(), p->degrees.end(), out); }

#define GTI_BIN(name, expr)                                                                     \
  int name(gtp_ctx* c, const gti_poly* a, const gti_poly* b, gti_poly** out) {                  \
    return wrap(c, [&] {                                                                        \
      GTP_CHECK(a && b && out, GTP_ERR_ARG, "null argument");                                   \
      *out = (expr).release();                                                                  \
    });                                                                                         \
  }
GTI_BIN(gti_add, poly_add(*c, *a, *b, false))
GTI_BIN(gti_sub, poly_add(*c, *a, *b, true))
GTI_BIN(gti_mul, poly_mul(*c, *a, *b))
GTI_BIN(gti_div, poly_div(*c, *a, *b))
#undef GTI_BIN
int gti_neg(gtp_ctx* c, const gti_poly* a, gti_poly** out) { return wrap(c, [&] { *out = poly_neg(*c, *a).release(); }); }
int gti_exp(gtp_ctx* c, const gti_poly* a, gti_poly** out) { return wrap(c, [&] { *out = poly_exp_log(*c, *a, false).release(); }); }
int gti_log(gtp_ctx* c, const gti_poly* a, gti_poly** out) { return wrap(c, [&] { *out = poly_exp_log(*c, *a, true).release(); }); }
int gti_pow(gtp_ctx* c, const gti_poly* a, uint32_t e, gti_poly** out) { return wrap(c, [&] { *out = poly_pow(*c, *a, e).release(); }); }
int gti_derivative(gtp_ctx* c, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out) { return wrap(c, [&] { *out = slice_scale(*c, *a, v, n, 0).release(); }); }
int gti_taylor_expansion_of_coeff(gtp_ctx* c, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out) {
  return wrap(c, [&] { *out = slice_scale(*c, *a, v, n, 1).release(); });
}
int gti_shift_down(gtp_ctx* c, const gti_poly* a, uint64_t v, uint64_t n, gti_poly** out) { return wrap(c, [&] { *out = poly_shift_down(*c, *a, v, n).release(); }); }
int gti_coefficients_of_term(gtp_ctx* c, const gti_poly* a, uint64_t v, uint64_t order, gti_poly** out) {   // :341-358
  return wrap(c, [&] {
    if (v >= a->shape.size()) { *out = (order == 0 ? share(*a) : scalar(*c, gti::iv(0.0, 0.0), a->degrees)).release(); return; }
    if (order >= a->shape[v]) { *out = scalar(*c, gti::iv(0.0, 0.0), a->degrees).release(); return; }
    Shape ext = a->shape, lo(a->shape.size(), 0);
    ext[v] = 1;
    lo[v] = order;
    *out = copy_box(*c, *a, lo, ext, a->degrees).release();
  });
}
int gti_taylor_polynomial_terms(gtp_ctx* c, const gti_poly* a, uint64_t v, const uint64_t* orders, int n_orders, gti_poly** out) {   // :380-404
  return wrap(c, [&] {
    u64 max_order_p1 = 1;
    bool has0 = false;
    for (int i = 0; i < n_orders; i++) {
      max_order_p1 = std::max(max_order_p1, orders[i] + 1);
      has0 |= orders[i] == 0;
    }
    if (v >= a->shape.size()) { *out = (has0 ? share(*a) : scalar(*c, gti::iv(0.0, 0.0), a->degrees)).release(); return; }
    const u64 upper = std::min(a->shape[v], max_order_p1);
    std::vector<unsigned char> keep(max_order_p1, 0);
    for (int i = 0; i < n_orders; i++) keep[orders[i]] = 1;
    BufP kb = c->alloc((max_order_p1 + 7) / 8 + 1);
    GTP_CUDA(cudaMemcpyAsync(kb->d, keep.data(), max_order_p1, cudaMemcpyHostToDevice, c->stream));
    c->sync();
    Shape ext = a->shape;
    ext[v] = upper;
    IvP r = fresh(*c, ext, a->degrees);
    Opnd A;
    A.p = a->ptr();
    A.shape = a->shape;
    ew(*c, EW_MASK, ext, A, nullptr, r->mptr(), ext, {}, (int)v, nullptr, (const unsigned char*)kb->d);
    *out = r.release();
  });
}
int gti_subst_var(gtp_ctx* c, const gti_poly* a, uint64_t v, const gti_poly* s, gti_poly** out) { return wrap(c, [&] { *out = poly_subst_var(*c, *a, v, *s).release(); }); }
int gti_truncate_to_degree_p1(gtp_ctx* c, const gti_poly* a, uint64_t d, gti_poly** out) {
  return wrap(c, [&] { *out = truncate_degrees(*c, *a, Shape(a->degrees.size(), d)).release(); });
}
int gti_remove_last_variable(gtp_ctx* c, const gti_poly* a, gti_poly** out) {   // :172-181
  return wrap(c, [&] {
    GTP_CHECK(!a->degrees.empty(), GTP_ERR_INDEX, "remove_last_variable on a 0-variable polynomial");
    const size_t v = a->degrees.size() - 1;
    Shape d(a->degrees.begin(), a->degrees.end() - 1), s(a->shape.begin(), a->shape.end() - 1);
    if (a->shape[v] == 1) {
      IvP r = mk(a->buf, a->off, s, d);
      r->known = a->known;
      r->first = a->first;
      *out = r.release();
      return;
    }
    Shape ext = a->shape;
    ext[v] = 1;
    IvP r = copy_box(*c, *a, Shape(ext.size(), 0), ext, a->degrees);
    *out = mk(r->buf, 0, s, d).release();
  });
}
int gti_extend_to_dim(gtp_ctx* c, const gti_poly* a, uint64_t ndim, uint64_t degree_p1, gti_poly** out) {   // :81-89
  return wrap(c, [&] {
    GTP_CHECK(a->shape.size() <= ndim && ndim <= (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "extend_to_dim: bad ndim");
    IvP r = share(*a);
    r->shape.resize(ndim, 1);
    r->degrees.resize(ndim, degree_p1);
    *out = r.release();
  });
}
int gti_constant_term(gtp_ctx* c, const gti_poly* a, double* out2) {
  return wrap(c, [&] {
    const Iv v = first_of(*c, *a);
    out2[0] = v.lo;
    out2[1] = v.hi;
  });
}
int gti_extract_constant(gtp_ctx* c, const gti_poly* a, int* is_constant, double* out2) {
  return wrap(c, [&] {
    *is_constant = a->len() == 1;
    if (*is_constant) {
      const Iv v = first_of(*c, *a);
      out2[0] = v.lo;
      out2[1] = v.hi;
    }
  });
}
int gti_gather_axis(gtp_ctx* c, const gti_poly* a, uint64_t v, uint64_t count, double* out_pairs) {
  return wrap(c, [&] {
    if (count == 0) return;
    const u64 len = v < a->shape.size() ? a->shape[v] : 1;
    u64 stride = 0;
    if (v < a->shape.size()) stride = strides_of(a->shape)[v];
    BufP tmp = c->alloc(2 * count);
    GTP_LAUNCH(*c, k_iv_gather, (unsigned)((count + 127) / 128), 128, 0, a->ptr(), stride, len, count, reinterpret_cast<Iv*>(tmp->d));
    GTP_CUDA(cudaMemcpyAsync(out_pairs, tmp->d, count * sizeof(Iv), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
  });
}

}  // extern "C"
