// C ABI of libgenfer_taylor: host-side shape algebra + operator dispatch of TaylorPoly<F64>
// (multivariate_taylor.rs) over the device kernels.  Shape logic follows the reference line by
// line (cited); all floating-point work happens on the device -- there is no CPU fallback.
#include <atomic>
#include <cmath>

#include "kernels.cuh"

using namespace gtp;
using PolyP = std::unique_ptr<gtp_poly>;

namespace gtp {

BufP Ctx::alloc(u64 n) {
  auto b = std::make_shared<Buf>();
  b->n = n;
  b->core = core;
  b->owned = true;
  const double t0 = hist ? now() : 0.0;
  const u64 cls = StreamCore::size_class(std::max<u64>(n, 1) * sizeof(double));
  b->cls_bytes = cls;
  b->d = (double*)core->take(cls);
  if (!b->d) {
    auto pool_alloc = [&]() {
      return core->pool ? cudaMallocFromPoolAsync((void**)&b->d, cls, core->pool, stream) : cudaMallocAsync((void**)&b->d, cls, stream);
    };
    cudaError_t e = pool_alloc();
    if (e == cudaErrorMemoryAllocation) {   // give the cached blocks back and try once more
      cudaGetLastError();
      core->trim();
      e = pool_alloc();
    }
    GTP_CUDA(e);
  }
  if (hist) t_alloc += now() - t0;
  if (!fused_cls.empty()) fused_cls.erase(b->d);   // a classification recorded for an earlier tensor at this address is stale
  return b;
}

BufP Ctx::alloc_host_visible(const double* vals, int n) {
  if (!scalars || n > 2) return nullptr;
  double* slot = scalars->acquire();
  if (!slot) return nullptr;
  for (int i = 0; i < n; i++) slot[i] = vals[i];
  auto b = std::make_shared<Buf>();
  b->d = slot;
  b->n = (u64)n;
  b->owned = false;
  b->core = core;
  b->pool = scalars;
  return b;
}

}  // namespace gtp

namespace {

// ---- shape algebra (multivariate_taylor.rs:114-170) -------------------------------------------
Shape min_degrees(const gtp_poly& a, const gtp_poly& b) {  // :114-127
  Shape d(std::max(a.degrees.size(), b.degrees.size()), UNB);
  for (size_t v = 0; v < d.size(); v++) {
    if (v < a.degrees.size()) d[v] = std::min(d[v], a.degrees[v]);
    if (v < b.degrees.size()) d[v] = std::min(d[v], b.degrees[v]);
  }
  return d;
}
Shape max_shape(const gtp_poly& a, const gtp_poly& b) {  // :129-148
  Shape s(std::max(a.shape.size(), b.shape.size()), 1);
  for (size_t v = 0; v < s.size(); v++) {
    if (v < a.shape.size()) s[v] = std::max(s[v], a.shape[v]);
    if (v < b.shape.size()) s[v] = std::max(s[v], b.shape[v]);
    if (v < a.degrees.size()) s[v] = std::min(s[v], a.degrees[v]);
    if (v < b.degrees.size()) s[v] = std::min(s[v], b.degrees[v]);
  }
  return s;
}
Shape sum_shape(const gtp_poly& a, const gtp_poly& b) {  // :150-170
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

void check_invariants(const Shape& shape, const Shape& degrees) {  // :23-31
  GTP_CHECK(shape.size() == degrees.size(), GTP_ERR_SHAPE, "coeffs.ndim() != degrees_p1.len()");
  GTP_CHECK(shape.size() <= (size_t)GTP_MAX_NDIM, GTP_ERR_ARG, "ndim exceeds GTP_MAX_NDIM");
  for (size_t i = 0; i < shape.size(); i++)
    GTP_CHECK(0 < shape[i] && shape[i] <= degrees[i], GTP_ERR_SHAPE, "need 0 < shape[i] <= degrees_p1[i]");
}

PolyP make_poly(BufP buf, u64 off, Shape shape, Shape degrees) {
  check_invariants(shape, degrees);
  PolyP p(new gtp_poly());
  p->buf = std::move(buf);
  p->off = off;
  p->shape = std::move(shape);
  p->degrees = std::move(degrees);
  return p;
}
// the buffer behind a handle (replicates a distributed tensor first)
BufP buf_of(const gtp_poly& a) {
  if (!a.shard) return a.buf;
  replicate(*a.shard);
  return a.shard->full;
}
PolyP share(const gtp_poly& a) {  // Clone: buffers are immutable, so sharing is a deep copy in effect
  PolyP p(new gtp_poly(a));
  return p;
}
PolyP new_zeros(Ctx& c, const Shape& shape, const Shape& degrees) {
  BufP b = c.alloc(prod(shape));
  GTP_CUDA(cudaMemsetAsync(b->d, 0, std::max<u64>(prod(shape), 1) * sizeof(double), c.stream));
  return make_poly(b, 0, shape, degrees);
}
PolyP new_uninit(Ctx& c, const Shape& shape, const Shape& degrees) {
  return make_poly(c.alloc(prod(shape)), 0, shape, degrees);
}
PolyP from_values(Ctx& c, const Shape& shape, const Shape& degrees, const double* host) {
  PolyP p = new_uninit(c, shape, degrees);
  GTP_CUDA(cudaMemcpyAsync(p->buf->d, host, prod(shape) * sizeof(double), cudaMemcpyHostToDevice, c.stream));
  // Pageable sources are staged by the driver before cudaMemcpyAsync returns; a PINNED source is read by the DMA engine
  // later, so the caller could overwrite or free it before the copy runs.  gtp_from_host promises "data may be reused on
  // return": wait for the copy when the source is pinned / registered host memory.
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host) != cudaSuccess) {
    cudaGetLastError();
    c.sync();
  } else if (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged) {
    c.sync();
  }
  return p;
}
PolyP scalar_poly(Ctx& c, double x, Shape shape_ones, Shape degrees) {
  PolyP p;
  if (BufP slot = c.alloc_host_visible(&x, 1)) {   // written by the host: no launch
    p = make_poly(slot, 0, shape_ones, degrees);
  } else {
    p = new_uninit(c, shape_ones, degrees);
    launch_fill(c, p->buf->d, 1, x);
  }
  p->cls->known = true;
  p->cls->linear = false;
  p->cls->first = x;
  return p;
}
PolyP zero_with(Ctx& c, const Shape& degrees) {  // :208-216
  return scalar_poly(c, 0.0, Shape(degrees.size(), 1), degrees);
}

// ---- data-dependent predicates (cached per handle) ----------------------------------------------
// The producing kernel may already have classified this tensor (fused_cls_begin): wait for its slot instead of launching.
static bool classify_from_producer(Ctx& c, const gtp_poly& p) {
  if (c.fused_cls.empty() || p.off != 0) return false;
  auto it = c.fused_cls.find(p.ptr());
  if (it == c.fused_cls.end() || it->second.shape != p.shape) return false;
  const unsigned long long seq = it->second.seq;
  if (c.cls_seq - seq >= Ctx::CLS_RING) return false;   // the ring has wrapped past this slot
  const ClsSlot* slot = c.cls_ring + (seq % Ctx::CLS_RING);
  const double t0 = c.hist ? Ctx::now() : 0.0;
  auto ready = [&] { return slot->seq_a == seq && slot->seq_b == (unsigned)seq; };
  for (unsigned long long spins = 0; !ready(); ++spins) {
    if (slot->seq_a > seq) return false;
    if ((spins & 0xfffff) == 0xfffff) {
      cudaError_t e = cudaStreamQuery(c.stream);
      if (e != cudaSuccess && e != cudaErrorNotReady) GTP_CUDA(e);
      if (e == cudaSuccess && !ready()) return false;
    }
  }
  if (c.hist) c.t_spin += Ctx::now() - t0;
  // seqlock read: payload between two reads of both sequence copies -- a torn 16-byte device store (not excluded by
  // the CUDA memory model on every host interconnect) shows up as a sequence mismatch on the second read and is retried
  double first, m;
  unsigned axis_p1;
  for (;;) {
    std::atomic_thread_fence(std::memory_order_acquire);
    first = slot->first;
    m = slot->m;
    axis_p1 = slot->axis_p1;
    std::atomic_thread_fence(std::memory_order_acquire);
    if (ready()) break;
    if (slot->seq_a > seq) return false;
  }
  p.cls->first = first;
  p.cls->linear = axis_p1 != 0;      // 1 + the first stored axis of length >= 2 that qualifies (:277-292)
  if (p.cls->linear) {
    p.cls->c = p.cls->first;
    p.cls->m = m;
    p.cls->v = axis_p1 - 1;
  }
  p.cls->known = true;
  c.fused_hits++;
  return true;
}
void classify(Ctx& c, const gtp_poly& p) {
  if (p.cls->known) return;
  if (classify_from_producer(c, p)) return;
  if (p.len() == 1) {
    if (!classify_small_zero_copy(c, p.ptr(), p.shape)) {
      GTP_CUDA(cudaMemcpyAsync(&c.rb_host->vals[0], p.ptr(), sizeof(double), cudaMemcpyDefault, c.stream));
      c.sync();
    }
    p.cls->first = c.rb_host->vals[0];
    p.cls->linear = false;
    p.cls->known = true;
    return;
  }
  if (!classify_small_zero_copy(c, p.ptr(), p.shape)) {
    launch_classify(c, p.ptr(), p.shape, c.rb_dev);
    GTP_CUDA(cudaMemcpyAsync(c.rb_host, c.rb_dev, offsetof(Readback, seq), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
  }
  p.cls->first = c.rb_host->vals[0];
  p.cls->linear = false;
  for (size_t v = 0; v < p.shape.size(); v++) {  // first axis of stored length >= 2 that qualifies (:277-292)
    if (p.shape[v] < 2) continue;
    if (!(c.rb_host->viol_mask & (1u << v))) {
      p.cls->linear = true;
      p.cls->c = p.cls->first;
      p.cls->m = c.rb_host->vals[1 + v];
      p.cls->v = v;
      break;
    }
  }
  p.cls->known = true;
}
bool is_zero(Ctx& c, const gtp_poly& p) {  // :643-645
  if (p.len() != 1) return false;
  classify(c, p);
  return p.cls->first == 0.0;
}
bool is_one(Ctx& c, const gtp_poly& p) {  // :653-655
  if (p.len() != 1) return false;
  classify(c, p);
  return p.cls->first == 1.0;
}

// ---- views / truncation --------------------------------------------------------------------------
u64 stride_of(const Shape& shape, size_t axis) {
  u64 s = 1;
  for (size_t i = axis + 1; i < shape.size(); i++) s *= shape[i];
  return s;
}

// Copy of the box [lo, lo+ext) of `a` as a new compact tensor.
PolyP copy_box(Ctx& c, const gtp_poly& a, const Shape& lo, const Shape& ext, const Shape& degrees) {
  PolyP r = new_uninit(c, ext, degrees);
  EwOperand A;
  A.p = a.ptr();
  A.shape = a.shape;
  A.lo = lo;
  launch_ew(c, EW_COPY, ext, A, nullptr, r->buf->d, ext, {});
  return r;
}

// truncate_degrees_p1 (:195-204): degrees = min(degrees, d); stored axes longer than d are cut.
PolyP truncate_degrees(Ctx& c, const gtp_poly& a, const Shape& d) {
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
    PolyP r = share(a);
    r->degrees = nd;
    return r;
  }
  if (!cut_inner) {  // only the leading axis shrinks: the result is a prefix of the same buffer
    PolyP r = make_poly(buf_of(a), a.off, ns, nd);
    return r;
  }
  return copy_box(c, a, Shape(ns.size(), 0), ns, nd);
}

// broadcast (:832-852): metadata only (trailing unit axes, trailing degrees of the other operand)
void broadcast(gtp_poly& x, gtp_poly& y) {
  if (x.degrees.size() < y.degrees.size()) x.degrees.insert(x.degrees.end(), y.degrees.begin() + x.degrees.size(), y.degrees.end());
  else if (y.degrees.size() < x.degrees.size()) y.degrees.insert(y.degrees.end(), x.degrees.begin() + y.degrees.size(), x.degrees.end());
  if (x.shape.size() < y.shape.size()) x.shape.resize(y.shape.size(), 1);
  if (y.shape.size() < x.shape.size()) y.shape.resize(x.shape.size(), 1);
}

PolyP with_degrees(PolyP p, const Shape& d) {
  p->degrees = d;
  check_invariants(p->shape, p->degrees);
  return p;
}

// element-wise op of a whole tensor against a device scalar
PolyP ew_scalar(Ctx& c, EwOp op, const gtp_poly& a, const gtp_poly& sp, const Shape& degrees) {
  PolyP r = new_uninit(c, a.shape, degrees);
  EwOperand A;
  A.p = a.ptr();
  A.shape = a.shape;
  // a scalar whose value the host already knows (constants, classified handles) travels in the kernel parameters
  const double* by_value = (sp.cls->known && sp.len() == 1) ? &sp.cls->first : nullptr;
  launch_ew(c, op, a.shape, A, nullptr, r->buf->d, a.shape, {}, -1, nullptr, nullptr, by_value ? nullptr : sp.ptr(), nullptr, 0, by_value);
  return r;
}

}  // namespace
namespace gtp { void partition_rows(u64 n_rows, int world, int rank, std::vector<u64>* out); }   // group.cu
namespace {
PolyP poly_add(Ctx& c, const gtp_poly& a0, const gtp_poly& b0, bool subtract);
PolyP poly_mul(Ctx& c, const gtp_poly& a0, const gtp_poly& b0);
PolyP poly_div(Ctx& c, const gtp_poly& a0, const gtp_poly& b0, PolyP* recip_cache = nullptr);
PolyP poly_recip(Ctx& c, const gtp_poly& y, const Shape& ws);

// ---- Add / Sub (:854-937) --------------------------------------------------------------------------
PolyP poly_add(Ctx& c, const gtp_poly& a0, const gtp_poly& b0, bool subtract) {
  Shape rd = min_degrees(a0, b0);
  gtp_poly a = a0, b = b0;
  broadcast(a, b);
  PolyP at = truncate_degrees(c, a, rd), bt = truncate_degrees(c, b, rd);
  if (bt->len() == 1)  // `*self.first_mut() (+|-)= other.first()` (:862-865, :919-922)
    return ew_scalar(c, subtract ? EW_SUB_FIRST : EW_ADD_FIRST, *at, *bt, rd);
  if (at->len() == 1)  // (:866-869) / `-(other - self)` (:923-926)
    return ew_scalar(c, subtract ? EW_RSUB_FIRST : EW_ADD_FIRST, *bt, *at, rd);
  Shape shape = max_shape(*at, *bt);
  PolyP r = new_uninit(c, shape, rd);
  EwOperand A, B;
  A.p = at->ptr();
  A.shape = at->shape;
  A.valid = at->shape;
  B.p = bt->ptr();
  B.shape = bt->shape;
  B.valid = bt->shape;
  launch_ew(c, subtract ? EW_SUB : EW_ADD, shape, A, &B, r->buf->d, shape, {});
  return r;
}

PolyP poly_neg(Ctx& c, const gtp_poly& a) {  // :902-909
  PolyP r = new_uninit(c, a.shape, a.degrees);
  EwOperand A;
  A.p = a.ptr();
  A.shape = a.shape;
  launch_ew(c, EW_NEG, a.shape, A, nullptr, r->buf->d, a.shape, {});
  return r;
}

// ---- mul_var / mul_linear (:589-623) ---------------------------------------------------------------
PolyP mul_var(Ctx& c, const gtp_poly& self, const double* m_dev, u64 v, const Shape& shape, const Shape& degrees) {
  u64 upper = std::min(shape[v] - 1, self.shape[v]);
  PolyP r = new_zeros(c, shape, degrees);
  Shape ext(self.shape.size());
  for (size_t a = 0; a < ext.size(); a++) ext[a] = std::min(self.shape[a], shape[a]);
  ext[v] = upper;
  if (prod(ext) == 0) return r;
  EwOperand A;
  A.p = self.ptr();
  A.shape = self.shape;
  Shape olo(shape.size(), 0);
  olo[v] = 1;
  launch_ew(c, EW_SCALE_DEV, ext, A, nullptr, r->buf->d, shape, olo, -1, nullptr, nullptr, m_dev);
  return r;
}
PolyP mul_linear(Ctx& c, const gtp_poly& self, double cst, double m, const double* m_dev, u64 v, const Shape& shape,
                 const Shape& degrees) {
  // One fused pass when the result keeps the shape of `self` on every other axis and neither side of the reference's
  // `mul_var(..) + self * c` would take a scalar fast path (those have their own rounding / signed-zero behaviour).
  bool fused = self.len() > 1 && prod(shape) > 1 && prod(shape) < (1ull << 32) - 4096 && shape.size() == self.shape.size() &&
               (shape[v] == self.shape[v] || shape[v] == self.shape[v] + 1) && c.fuse_mul_linear;
  for (size_t a = 0; fused && a < shape.size(); a++)
    if (a != v && shape[a] != self.shape[a]) fused = false;
  if (fused) {
    PolyP r = new_uninit(c, shape, degrees);
    u64 outer = 1, inner = 1;
    for (size_t a = 0; a < v; a++) outer *= shape[a];
    for (size_t a = v + 1; a < shape.size(); a++) inner *= shape[a];
    launch_mul_linear(c, self.ptr(), r->buf->d, outer, self.shape[v], shape[v], inner, cst, m, shape);
    return r;
  }
  if (cst == 0.0) return mul_var(c, self, m_dev, v, shape, degrees);
  PolyP shifted = mul_var(c, self, m_dev, v, shape, degrees);
  PolyP cpoly = scalar_poly(c, cst, {}, {});
  PolyP scaled = poly_mul(c, self, *cpoly);
  return poly_add(c, *shifted, *scaled, false);
}

// ---- Mul (:1014-1072) --------------------------------------------------------------------------------
PolyP poly_mul(Ctx& c, const gtp_poly& a0, const gtp_poly& b0) {
  Shape d = min_degrees(a0, b0);
  if (is_zero(c, a0) || is_zero(c, b0)) return zero_with(c, d);  // :1021-1023
  gtp_poly a = a0, b = b0;
  broadcast(a, b);
  Shape shape = sum_shape(a, b);  // from the pre-truncation stored shapes (:1027)
  PolyP at = truncate_degrees(c, a, d), bt = truncate_degrees(c, b, d);
  if (is_one(c, *at)) return with_degrees(share(*bt), d);  // :1032-1037
  if (is_one(c, *bt)) return with_degrees(share(*at), d);
  if (at->len() == 1) return ew_scalar(c, EW_SCALE_DEV, *bt, *at, d);  // :1040-1043  c * x
  if (bt->len() == 1) return ew_scalar(c, EW_SCALE_DEV, *at, *bt, d);  // :1044-1047
  classify(c, *at);
  if (at->cls->linear) {  // :1052-1056
    u64 v = at->cls->v;
    Shape s = bt->shape;
    s[v] = std::min(d[v], s[v] + 1);
    return mul_linear(c, *bt, at->cls->c, at->cls->m, at->ptr() + stride_of(at->shape, v), v, s, d);
  }
  classify(c, *bt);
  if (bt->cls->linear) {  // :1057-1061
    u64 v = bt->cls->v;
    Shape s = at->shape;
    s[v] = std::min(d[v], s[v] + 1);
    return mul_linear(c, *at, bt->cls->c, bt->cls->m, bt->ptr() + stride_of(bt->shape, v), v, s, d);
  }
  // general case (:1064-1070)
  // (threshold 0 partitions every general product, also on a one-rank group: single-GPU tests of this path)
  if (c.group && (c.group->world > 1 || c.group->threshold == 0) && shape.size() >= 2 && prod(shape) >= c.group->threshold &&
      shape[0] >= 2 * (u64)c.group->world) {
    // Partitioned product (SURVEY 8e): this rank computes its folded-cyclic leading-axis rows; the result stays
    // row-sharded until somebody needs all of it.  Both operands are read whole (replicated on first use).
    auto sh = std::make_shared<ShardState>();
    sh->kind = ShardState::ROWS;
    sh->ctx = &c;
    sh->group = c.group;
    partition_rows(shape[0], c.group->world, c.group->rank, &sh->rows);
    sh->n_rows = shape[0];
    sh->row_elems = prod(shape) / shape[0];
    sh->local = c.alloc(std::max<u64>(sh->rows.size() * sh->row_elems, 1));
    MulArgs m;
    m.ndim = (int)shape.size();
    m.xs = at->shape;
    m.ys = bt->shape;
    m.rs = shape;
    m.x = at->ptr();
    m.y = bt->ptr();
    m.out = sh->local->d;
    m.rows = sh->rows;
    if (!m.rows.empty()) launch_mul(c, m);
    c.group->partitioned_products++;
    PolyP r = make_poly(nullptr, 0, shape, d);
    r->shard = sh;
    return r;
  }
  PolyP r = new_uninit(c, shape, d);
  MulArgs m;
  m.ndim = (int)shape.size();
  m.xs = at->shape;
  m.ys = bt->shape;
  m.rs = shape;
  m.x = at->ptr();
  m.y = bt->ptr();
  m.out = r->buf->d;
  m.row_begin = 0;
  m.row_step = 1;
  m.row_count = shape.empty() ? 1 : shape[0];
  launch_mul(c, m);
  return r;
}

// ---- Div (:1194-1231) ----------------------------------------------------------------------------------
PolyP poly_div(Ctx& c, const gtp_poly& a0, const gtp_poly& b0, PolyP* recip_cache) {
  gtp_poly a = a0, b = b0;
  broadcast(a, b);
  Shape d = min_degrees(a, b);  // after broadcast (:1199-1200)
  PolyP at = truncate_degrees(c, a, d), bt = truncate_degrees(c, b, d);
  if (is_one(c, *bt)) return with_degrees(share(*at), d);                     // :1205-1207
  if (bt->len() == 1) return ew_scalar(c, EW_DIV_DEV, *at, *bt, d);     // :1210-1213
  Shape rs = d;
  int nonunit = 0, axis = -1;
  for (size_t i = 0; i < rs.size(); i++) {
    if (bt->shape[i] == 1) rs[i] = at->shape[i];  // :1216-1221
    else { nonunit++; axis = (int)i; }
  }
  for (u64 x : rs) GTP_CHECK(x != UNB, GTP_ERR_SHAPE, "division by a non-constant series needs bounded degrees");
  PolyP r = new_uninit(c, rs, d);
  if (nonunit == 1) {
    u64 outer = 1, inner = 1;
    for (int i = 0; i < axis; i++) outer *= rs[i];
    for (size_t i = axis + 1; i < rs.size(); i++) inner *= rs[i];
    launch_div_axis(c, at->ptr(), bt->ptr(), r->buf->d, outer, inner, at->shape[axis], bt->shape[axis], rs[axis],
                    at->shape, rs, axis);
  } else if (c.fast_mul == 0) {
    launch_div_general(c, at->ptr(), at->shape, bt->ptr(), bt->shape, r->buf->d, rs);   // exact-order mode: wavefront kernel
  } else if (c.use_wave && launch_rec_wave(c, 0, at->ptr(), at->shape, bt->ptr(), bt->shape, r->buf->d, rs, false)) {
    // the reference's recurrence (:1170-1191) as one device-resident kernel
  } else {
    // x / y = x (*) (1 / y): the reciprocal series costs 2 products per slice of every non-unit axis (recip_rec), all of
    // them on the product kernels; the wavefront kernel keeps a few thousand threads busy and is slower than one host
    // core beyond ~10^4 coefficients.  Same value in exact arithmetic, tolerance-checked like the DFMA products.
    Shape ws = rs;
    for (size_t i = 0; i < ws.size(); i++)
      if (bt->shape[i] == 1) ws[i] = 1;
    PolyP w = (recip_cache && *recip_cache) ? share(**recip_cache) : poly_recip(c, *bt, ws);
    if (recip_cache && !*recip_cache) *recip_cache = share(*w);
    MulArgs m;
    m.ndim = (int)rs.size();
    m.xs = at->shape;
    m.ys = ws;
    m.rs = rs;
    m.x = at->ptr();
    m.y = w->ptr();
    m.out = r->buf->d;
    m.row_begin = 0;
    m.row_step = 1;
    m.row_count = rs.empty() ? 1 : rs[0];
    launch_mul(c, m);
  }
  return r;
}

// ---- exp / log (:406-430, :1271-1386) ------------------------------------------------------------------
bool one_d_len(const Shape& s, size_t from, u64* n) {  // extract_1d_len (:958-969) on shape[from..]
  bool found = false;
  for (size_t i = from; i < s.size(); i++) {
    if (s[i] != 1) {
      if (found) return false;
      found = true;
      *n = s[i];
    }
  }
  return found;
}
u64 tail_prod(const Shape& s, size_t from) {
  u64 p = 1;
  for (size_t i = from; i < s.size(); i++) p *= s[i];
  return p;
}
Shape tail(const Shape& s, size_t from) { return Shape(s.begin() + from, s.end()); }

// ---- reciprocal series (for the general Div) ---------------------------------------------------------------
// W = 1 / Y on the sub-views ys[from..] / ws[from..]:  W[0] = 1 / Y[0] (one axis less);
// W[k] = -(sum_{j<k} W[j] (*) Y[k-j]) (*) W[0]   -- the reference's div recurrence (:1170-1191) for X = 1 with the inner
// division by Y[0] replaced by a product with its reciprocal.  ws[i] == 1 wherever Y is constant along axis i.
void recip_rec(Ctx& c, const double* yp, const Shape& ys, double* wp, const Shape& ws, size_t from, const double* one_dev) {
  const size_t nd = ws.size();
  int nonunit = 0, axis = -1;
  for (size_t i = from; i < nd; i++)
    if (ws[i] != 1) { nonunit++; axis = (int)i; }
  if (nonunit <= 1) {   // scalar or one varying axis: the single-axis division kernel with X = 1 (bit-exact recurrence)
    const u64 rl = nonunit ? ws[axis] : 1, yl = nonunit ? ys[axis] : 1;
    Shape one_shape(nd - from, 1), w_shape = tail(ws, from);
    launch_div_axis(c, one_dev, yp, wp, 1, 1, 1, yl, rl, one_shape, w_shape, nonunit ? axis - (int)from : 0);
    return;
  }
  const u64 ystr = tail_prod(ys, from + 1), wstr = tail_prod(ws, from + 1);
  recip_rec(c, yp, ys, wp, ws, from + 1, one_dev);
  const u64 yl = ys[from], wl = ws[from];
  if (wl <= 1) return;
  BufP tmp = c.alloc(std::max<u64>(wstr, 1));
  Shape sub = tail(ws, from + 1);
  for (u64 k = 1; k < wl; k++) {
    double* cur = wp + k * wstr;
    if (yl <= 1) {
      GTP_CUDA(cudaMemsetAsync(cur, 0, wstr * sizeof(double), c.stream));
      continue;
    }
    // S = sum_{j<k} W[j] (*) Y[k-j] = leading-axis row k-1 of Y[1..] (*) W[0..k)
    MulArgs m;
    m.ndim = (int)(nd - from);
    m.xs = tail(ys, from);
    m.xs[0] = yl - 1;
    m.ys = tail(ws, from);
    m.ys[0] = k;
    m.rs = tail(ws, from);
    m.x = yp + ystr;
    m.y = wp;
    m.out = tmp->d;
    m.row_begin = k - 1;
    m.row_step = 1;
    m.row_count = 1;
    launch_mul(c, m);
    // W[k] = -(S (*) W[0])
    MulArgs q;
    q.ndim = (int)sub.size();
    q.xs = sub;
    q.ys = sub;
    q.rs = sub;
    q.x = tmp->d;
    q.y = wp;
    q.out = cur;
    q.row_begin = 0;
    q.row_step = 1;
    q.row_count = sub.empty() ? 1 : sub[0];
    launch_mul(c, q);
    launch_scale_const(c, cur, cur, wstr, -1.0, false);
  }
}
PolyP poly_recip(Ctx& c, const gtp_poly& y, const Shape& ws) {
  PolyP one = scalar_poly(c, 1.0, {}, {});
  PolyP w = new_uninit(c, ws, ws);
  recip_rec(c, y.ptr(), y.shape, w->buf->d, ws, 0, one->ptr());
  return w;
}

// exp (:1285-1317) on the sub-views xs[from..] / res[from..] located at xp / rp
void exp_rec(Ctx& c, const double* xp, const Shape& xs, double* rp, const Shape& rs, size_t from, const double* seed = nullptr) {
  if (tail_prod(xs, from) == 0) return;
  if (from == rs.size()) {  // res.ndim() == 0
    launch_scalar_fn(c, 0, xp, rp, seed);
    return;
  }
  u64 n;
  if (one_d_len(rs, from, &n)) {  // exp_1d on the flattened argument
    launch_exp_1d(c, xp, tail_prod(xs, from), rp, n, seed);
    return;
  }
  const u64 xstr = tail_prod(xs, from + 1), rstr = tail_prod(rs, from + 1);
  exp_rec(c, xp, xs, rp, rs, from + 1, seed);
  const u64 xl = xs[from], rl = rs[from];
  if (rl <= 1) return;
  // XS[j-1] = xs[j] * j for j = 1..xl-1  (`x * T::from(j)`, :1309)
  BufP scaled;
  if (xl > 1) {
    scaled = c.alloc((xl - 1) * xstr);
    launch_scale_rows(c, xp + xstr, scaled->d, xl - 1, xstr, 1, false);
  }
  for (u64 k = 1; k < rl; k++) {
    double* cur = rp + k * rstr;
    u64 hi = std::min(xl, k + 1);
    if (hi <= 1) {
      GTP_CUDA(cudaMemsetAsync(cur, 0, rstr * sizeof(double), c.stream));
    } else {
      // current = sum_{j=1}^{hi-1} XS[j] (*) res[k-j]  == leading-axis row k-1 of XS[1..] (*) res[0..k)
      MulArgs m;
      m.ndim = (int)(rs.size() - from);
      m.xs = tail(xs, from);
      m.xs[0] = xl - 1;
      m.ys = tail(rs, from);
      m.ys[0] = k;
      m.rs = tail(rs, from);
      m.x = scaled->d;
      m.y = rp;
      m.out = cur;
      m.row_begin = k - 1;
      m.row_step = 1;
      m.row_count = 1;
      launch_mul(c, m);
    }
    launch_scale_const(c, cur, cur, rstr, (double)k, true);  // current /= k (:1315)
  }
}

// log (:1335-1386)
void log_rec(Ctx& c, const double* xp, const Shape& xs, double* rp, const Shape& rs, size_t from, const double* seed = nullptr) {
  if (tail_prod(xs, from) == 0) return;
  if (from == rs.size()) {
    launch_scalar_fn(c, 1, xp, rp, seed);
    return;
  }
  u64 n;
  if (one_d_len(xs, from, &n)) {  // :1343 -- triggers on the ARGUMENT being 1-d
    u64 rn;
    GTP_CHECK(one_d_len(rs, from, &rn), GTP_ERR_SHAPE, "log: result of a 1-d argument is not 1-d");
    launch_log_1d(c, xp, tail_prod(xs, from), rp, rn, seed);
    return;
  }
  const u64 xstr = tail_prod(xs, from + 1), rstr = tail_prod(rs, from + 1);
  log_rec(c, xp, xs, rp, rs, from + 1, seed);
  const u64 xl = xs[from], rl = rs[from];
  if (rl <= 1) return;
  Shape cur_shape = tail(rs, from + 1), x_sub = tail(xs, from + 1);
  // RS[j] = res[j] * j  (:1362-1365), filled as rows become final; row 0 unused
  BufP rscaled = c.alloc(rl * rstr);
  BufP xk_scaled = c.alloc(std::max<u64>(xstr, 1));
  // the divisor xs[0] as a polynomial of degrees = current.shape (:1378-1381)
  PolyP den = make_poly(nullptr, 0, x_sub, cur_shape);
  {
    auto b = std::make_shared<Buf>();
    b->d = const_cast<double*>(xp);
    b->n = xstr;
    b->owned = false;
    den->buf = b;
  }
  PolyP den_recip;
  for (u64 k = 1; k < rl; k++) {
    double* cur = rp + k * rstr;
    u64 lo = std::max<u64>(sat_sub(k + 1, xl), 1);
    PolyP num = new_uninit(c, cur_shape, cur_shape);
    if (lo >= k) {
      GTP_CUDA(cudaMemsetAsync(num->buf->d, 0, std::max<u64>(rstr, 1) * sizeof(double), c.stream));
    } else {
      // sum_{j=lo}^{k-1} xs[k-j] (*) RS[j]: first operand xs[1..] (index a = k-j, visited DESCENDING as j
      // ascends), second RS[1..k); output row k-2 of xs[1..] (*) RS[1..k)
      MulArgs m;
      m.ndim = (int)(rs.size() - from);
      m.xs = tail(xs, from);
      m.xs[0] = xl - 1;
      m.ys = tail(rs, from);
      m.ys[0] = k - 1;
      m.rs = tail(rs, from);
      m.x = xp + xstr;
      m.y = rscaled->d + rstr;
      m.out = num->buf->d;
      m.row_begin = k - 2;
      m.row_step = 1;
      m.row_count = 1;
      launch_mul(c, m);
    }
    // current = -current; current[..xs_k] += k * xs_k  (:1369-1375)
    PolyP neg = poly_neg(c, *num);
    PolyP numer = std::move(neg);
    if (k < xl) {
      launch_scale_const(c, xp + k * xstr, xk_scaled->d, xstr, (double)k, false);
      PolyP xk = make_poly(nullptr, 0, x_sub, cur_shape);
      auto b = std::make_shared<Buf>();
      b->d = xk_scaled->d;
      b->n = xstr;
      b->owned = false;
      xk->buf = b;
      // zero-extended add into the leading block (slice_each_axis_mut(..).add_assign)
      PolyP sum = new_uninit(c, cur_shape, cur_shape);
      EwOperand A, B;
      A.p = numer->ptr();
      A.shape = cur_shape;
      A.valid = cur_shape;
      B.p = xk->ptr();
      B.shape = x_sub;
      B.valid = x_sub;
      // reference adds into existing values: cur + xk (no leading 0 +): emulate with ADD where A is
      // always valid; (0 + a) + b equals a + b except for a = -0.0, b absent -- harmless here.
      launch_ew(c, EW_ADD, cur_shape, A, &B, sum->buf->d, cur_shape, {});
      numer = std::move(sum);
    }
    PolyP q = poly_div(c, *numer, *den, &den_recip);  // full Div dispatch (:1376-1383); 1 / xs[0] is computed once
    GTP_CHECK(q->shape == cur_shape, GTP_ERR_SHAPE, "log: quotient shape mismatch");
    launch_scale_const(c, q->ptr(), cur, rstr, (double)k, true);                 // current /= k (:1384)
    launch_scale_const(c, cur, rscaled->d + k * rstr, rstr, (double)k, false);    // RS[k] = res[k] * k
  }
}

PolyP poly_exp_log(Ctx& c, const gtp_poly& a, bool is_log) {
  Shape rs = a.degrees;
  for (size_t i = 0; i < rs.size(); i++)
    if (a.shape[i] == 1) rs[i] = 1;  // :408-413 / :421-426
  for (u64 x : rs) GTP_CHECK(x != UNB, GTP_ERR_SHAPE, "exp/log of a non-constant series needs bounded degrees");
  // The one transcendental of the call -- exp / log of the constant term (:1273, :1290, :1321, :1340) -- is taken from
  // the host's libm whenever the host knows the constant term (small tensors carry it in their cached classification):
  // that is the function the reference calls, so the seed is bit-identical.  Large tensors use CUDA's <= 1 ulp exp / log
  // on the device instead of synchronising.
  double seed_val = 0.0;
  const double* seed = nullptr;
  if (a.len() <= 8192) {
    classify(c, a);
    seed_val = is_log ? std::log(a.cls->first) : std::exp(a.cls->first);
    seed = &seed_val;
  }
  if (c.use_wave && c.fast_mul != 0) {
    // N-D (two or more non-unit axes): the whole recurrence in one cooperative kernel.  Small exp calls (the
    // reference-order product kernel would have served their inner sums) run its exact-order mode and stay bit-identical.
    int nonunit = 0;
    for (u64 x : rs) nonunit += x > 1;
    const bool small = mul_macs(a.shape, rs, rs) < DFMA_MIN_MACS;
    if (nonunit >= 2) {
      PolyP r = new_uninit(c, rs, a.degrees);
      if (launch_rec_wave(c, is_log ? 2 : 1, a.ptr(), a.shape, nullptr, Shape(), r->buf->d, rs, !is_log && small, seed)) return r;
    }
  }
  PolyP r = new_zeros(c, rs, a.degrees);
  if (is_log) log_rec(c, a.ptr(), a.shape, r->buf->d, rs, 0, seed);
  else exp_rec(c, a.ptr(), a.shape, r->buf->d, rs, 0, seed);
  return r;
}

// ---- gathers along one axis ------------------------------------------------------------------------------
// slice n.. along v, scaled slice-wise by a device factor table of `kind` (derivative / coeff expansion)
PolyP slice_scale(Ctx& c, const gtp_poly& a, u64 v, u64 n, int kind) {
  GTP_CHECK(v < a.degrees.size() && n < a.degrees[v], GTP_ERR_INDEX, "variable / order out of range");  // :459, :486
  Shape d = a.degrees;
  d[v] = sat_sub(d[v], n);  // :467, :494
  if (n >= a.shape[v]) return zero_with(c, d);
  Shape ext = a.shape, lo(a.shape.size(), 0);
  ext[v] = a.shape[v] - n;
  lo[v] = n;
  PolyP r = new_uninit(c, ext, d);
  EwOperand A;
  A.p = a.ptr();
  A.shape = a.shape;
  A.lo = lo;
  double tab[1024];
  if (prod(ext) < (1ull << 32) - 4096 && host_factors(kind, n, ext[v], tab)) {   // one launch: the table rides in the parameters
    launch_ew(c, EW_COPY, ext, A, nullptr, r->buf->d, ext, {}, (int)v, nullptr, nullptr, nullptr, tab, (int)ext[v]);
    return r;
  }
  BufP fac = c.alloc(ext[v]);
  launch_factors(c, kind, n, ext[v], nullptr, fac->d);
  launch_ew(c, EW_COPY, ext, A, nullptr, r->buf->d, ext, {}, (int)v, fac->d);
  return r;
}

PolyP poly_shift_down(Ctx& c, const gtp_poly& a, u64 v, u64 n) {  // :514-536
  GTP_CHECK(v < a.degrees.size() && n < a.degrees[v], GTP_ERR_INDEX, "shift_down: variable / order out of range");
  Shape d = a.degrees;
  d[v] = sat_sub(d[v], n);
  Shape rs = a.shape;
  rs[v] = (a.shape[v] <= n + 1) ? 1 : a.shape[v] - n;
  PolyP r = new_uninit(c, rs, d);
  u64 outer = 1, inner = 1;
  for (size_t i = 0; i < v; i++) outer *= a.shape[i];
  for (size_t i = v + 1; i < a.shape.size(); i++) inner *= a.shape[i];
  launch_shift_down(c, a.ptr(), r->buf->d, outer, a.shape[v], inner, n, v + 1 == a.shape.size());
  return r;
}

PolyP poly_subst_var(Ctx& c, const gtp_poly& self, u64 v, const gtp_poly& subst) {  // :540-580
  if (v >= self.shape.size()) return share(self);
  Shape d = min_degrees(self, subst);
  if (is_zero(c, subst)) {  // :547-554
    Shape ext = self.shape, lo(self.shape.size(), 0);
    ext[v] = 1;
    Shape dd = d;
    if (ext.size() < dd.size()) ext.resize(dd.size(), 1);
    gtp_poly s2 = self;
    s2.shape.resize(ext.size(), 1);
    lo.resize(ext.size(), 0);
    return copy_box(c, s2, lo, ext, dd);
  }
  classify(c, subst);
  if (subst.cls->linear && subst.cls->v == v && subst.cls->c == 0.0) {  // :555-568
    GTP_CHECK(d.size() == self.shape.size(), GTP_ERR_SHAPE, "subst_var: substitution has more variables than self");
    Shape ext(self.shape.size());
    for (size_t a = 0; a < ext.size(); a++) ext[a] = std::min(self.shape[a], d[a]);
    PolyP r = new_uninit(c, ext, d);
    EwOperand A;
    A.p = self.ptr();
    A.shape = self.shape;
    double tab[1024];
    if (prod(ext) < (1ull << 32) - 4096 && host_factors(2, 0, ext[v], tab, subst.cls->m)) {   // m is known from the classification
      launch_ew(c, EW_COPY, ext, A, nullptr, r->buf->d, ext, {}, (int)v, nullptr, nullptr, nullptr, tab, (int)ext[v]);
      return r;
    }
    BufP fac = c.alloc(ext[v]);
    launch_factors(c, 2, 0, ext[v], subst.ptr() + stride_of(subst.shape, v), fac->d);
    launch_ew(c, EW_COPY, ext, A, nullptr, r->buf->d, ext, {}, (int)v, fac->d);
    return r;
  }
  // Horner from the highest stored slice (:569-579)
  PolyP res = zero_with(c, d);
  gtp_poly cs = self;
  cs.shape.resize(std::max(cs.shape.size(), d.size()), 1);
  Shape ext(cs.shape.size()), lo(cs.shape.size(), 0);
  for (size_t a = 0; a < ext.size(); a++) ext[a] = std::min(cs.shape[a], d[a]);
  GTP_CHECK(d[v] >= 1, GTP_ERR_SHAPE, "subst_var: zero degree along the substituted axis");
  ext[v] = 1;
  gtp_poly sb = subst;   // the substitution on the common axes (trailing unit axes, like broadcast :832-852)
  sb.shape.resize(cs.shape.size(), 1);
  for (u64 i = cs.shape[v]; i-- > 0;) {
    // Once res has grown past a scalar the rest of the loop is one fused kernel (kernels_horner.cu).  Mul's linear fast
    // path (:1052-1061) gives the general product's values but clips the stored shape to the other operand's (+1 along the
    // axis) when the linear operand carries explicit zeros: the fused loop is entered only with a non-linear Horner value
    // and a substitution that is non-linear or compactly linear (stored shape 2 along its axis, 1 elsewhere), where the
    // two paths also agree on the stored shape.
    if (c.use_horner && c.fast_mul != 0 && res->len() > 1 && sb.len() >= 2 && sb.len() <= 32 && res->shape.size() == cs.shape.size()) {
      bool subst_ok = !subst.cls->linear || sb.len() == 2;
      if (subst_ok) {
        classify(c, *res);
        if (!res->cls->linear) {
          BufP ob;
          Shape os;
          if (launch_horner(c, cs.ptr(), cs.shape, v, d, sb.ptr(), sb.shape, res->ptr(), res->shape, i, &ob, &os))
            return make_poly(ob, 0, os, d);
        }
      }
    }
    lo[v] = i;
    PolyP slice = copy_box(c, cs, lo, ext, d);
    PolyP prod_ = poly_mul(c, *res, subst);
    res = poly_add(c, *prod_, *slice, false);
  }
  return res;
}

PolyP poly_pow(Ctx& c, const gtp_poly& a, uint32_t e) {  // :433-451
  if (e == 0) return scalar_poly(c, 1.0, {}, {});
  if (e == 1) return share(a);
  PolyP res = scalar_poly(c, 1.0, {}, {});
  PolyP base = share(a);
  while (e > 0) {
    if (e & 1) res = poly_mul(c, *res, *base);
    base = poly_mul(c, *base, *base);  // also after the last bit (:447)
    e >>= 1;
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

}  // namespace

// ==================================================================================================
// C ABI
// ==================================================================================================
extern "C" {

int gtp_ctx_create(int device, void* cuda_stream, gtp_ctx** out) {
  if (!out) return GTP_ERR_ARG;
  *out = nullptr;
  static thread_local std::string create_err;
  gtp_ctx* c = new gtp_ctx();
  if (const char* h = getenv("GTP_LAUNCH_HIST"))
    if (h[0] == '1') c->hist = new std::map<std::string, u64>();
  int rc = wrap(c, [&] {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    GTP_CHECK(e == cudaSuccess && n > 0, GTP_ERR_CUDA,
              std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(e));
    GTP_CHECK(device >= 0 && device < n, GTP_ERR_ARG, "device index out of range");
    c->device = device;
    GTP_CUDA(cudaSetDevice(device));
    c->core = std::make_shared<StreamCore>();
    c->core->device = device;
    if (cuda_stream) {
      c->core->stream = (cudaStream_t)cuda_stream;
      c->core->own = false;
    } else {
      GTP_CUDA(cudaStreamCreateWithFlags(&c->core->stream, cudaStreamNonBlocking));
      c->core->own = true;
    }
    c->stream = c->core->stream;
    if (!(getenv("GTP_NO_FUSED_CLS") && getenv("GTP_NO_FUSED_CLS")[0] == '1')) {
      ClsSlot* ring = nullptr;
      if (cudaHostAlloc((void**)&ring, sizeof(ClsSlot) * Ctx::CLS_RING, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
        void* dp = nullptr;
        if (cudaHostGetDevicePointer(&dp, ring, 0) == cudaSuccess && dp == (void*)ring) {
          memset(ring, 0, sizeof(ClsSlot) * Ctx::CLS_RING);
          c->cls_ring = ring;
        } else {
          cudaGetLastError();
          cudaFreeHost(ring);
        }
      } else {
        cudaGetLastError();
      }
    }
    if (!(getenv("GTP_NO_SCALAR_POOL") && getenv("GTP_NO_SCALAR_POOL")[0] == '1')) {
      c->scalars = std::make_shared<ScalarPool>();
      c->scalars->core = c->core;
    }
    cudaDeviceProp prop;
    GTP_CUDA(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    // A PRIVATE stream-ordered pool that keeps freed blocks instead of returning them to the driver: the device's default
    // pool (shared with torch / NCCL allocations of the same process) is left untouched; gtp_ctx_trim() gives the memory back.
    {
      cudaMemPoolProps props;
      memset(&props, 0, sizeof(props));
      props.allocType = cudaMemAllocationTypePinned;
      props.handleTypes = cudaMemHandleTypeNone;
      props.location.type = cudaMemLocationTypeDevice;
      props.location.id = device;
      if (cudaMemPoolCreate(&c->core->pool, &props) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        GTP_CUDA(cudaMemPoolSetAttribute(c->core->pool, cudaMemPoolAttrReleaseThreshold, &thr));
      } else {
        cudaGetLastError();
        c->core->pool = nullptr;   // fall back to the default pool with its default (release-at-sync) threshold
      }
    }
    GTP_CUDA(cudaHostAlloc((void**)&c->rb_host, sizeof(Readback), cudaHostAllocMapped | cudaHostAllocPortable));
    memset(c->rb_host, 0, sizeof(Readback));
    if (cudaHostGetDevicePointer((void**)&c->rb_host_dev, c->rb_host, 0) != cudaSuccess) {
      c->rb_host_dev = nullptr;   // no zero-copy: classify() falls back to the copy + synchronise path
      cudaGetLastError();
    }
    GTP_CUDA(cudaMalloc((void**)&c->rb_dev, sizeof(Readback)));
    GTP_CUDA(cudaMemset(c->rb_dev, 0, sizeof(Readback)));
  });
  if (rc != GTP_OK) {
    fprintf(stderr, "gtp_ctx_create: %s\n", c->err.c_str());
    delete c;
    return rc;
  }
  if (const char* fm = getenv("GTP_FAST_MUL")) gtp_ctx_set_fast_mul(c, atoi(fm));   // A/B measurements of whole programs
  if (const char* dc = getenv("GTP_DIRECT_CTAS")) c->direct_ctas = std::max(1, atoi(dc));
  if (const char* dm = getenv("GTP_DIRECT_MIN")) c->direct_min = (u64)std::max(1ll, atoll(dm));
  *out = c;
  return GTP_OK;
}

void gtp_ctx_destroy(gtp_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->hist) {
    fprintf(stderr, "[gtp launches] %10llu  classifications served by the producing kernel\n", (unsigned long long)c->fused_hits);
    fprintf(stderr, "[gtp host time] launch calls %.3f s, cudaMallocAsync %.3f s, waiting for producer classifications %.3f s\n", c->t_launch, c->t_alloc, c->t_spin);
    for (auto& kv : *c->hist) fprintf(stderr, "[gtp launches] %10llu  %s\n", (unsigned long long)kv.second, kv.first.c_str());
    delete c->hist;
  }
  if (c->cls_ring) cudaFreeHost(c->cls_ring);
  if (c->rb_host) cudaFreeHost(c->rb_host);
  if (c->rb_dev) cudaFree(c->rb_dev);
  if (c->gather_host) cudaFreeHost(c->gather_host);
  delete c;
}
const char* gtp_last_error(gtp_ctx* c) { return c ? c->err.c_str() : "null context"; }
int gtp_ctx_synchronize(gtp_ctx* c) { return wrap(c, [&] { c->sync(); }); }
int gtp_ctx_trim(gtp_ctx* c) {   // give the cached free blocks back to the driver (other allocators of the process can use them)
  return wrap(c, [&] {
    c->core->trim();
    c->sync();
    if (c->core->pool) GTP_CUDA(cudaMemPoolTrimTo(c->core->pool, 0));
  });
}
void* gtp_ctx_stream(gtp_ctx* c) { return c ? (void*)c->stream : nullptr; }
uint64_t gtp_ctx_launch_count(gtp_ctx* c) { return c ? c->launches : 0; }
int gtp_ctx_set_fast_mul(gtp_ctx* c, int enabled) {
  if (!c) return GTP_ERR_ARG;
  // bits 4 and 8 are ignored (they selected the blocked kernel's retired table variants)
  c->use_slide = (enabled & 16) == 0;
  c->fuse_mul_linear = (enabled & 128) == 0;
  c->use_stencil = (enabled & 256) == 0;
  c->use_wave = (enabled & 1024) == 0;
  c->use_horner = (enabled & 2048) == 0;
  c->use_axis = (enabled & 4096) == 0;
  c->use_pad = (enabled & 8192) == 0;
  c->use_bulk = (enabled & 16384) == 0;
  c->bulk_products = (enabled & 32768) != 0;
  c->use_direct = (enabled & 65536) == 0;
  c->direct_products = (enabled & 131072) == 0;
  c->direct_products_all = (enabled & 262144) != 0;
  c->slide_runs = (enabled & 524288) == 0;
  c->stencil_v4 = (enabled & 512) == 0;
  c->slide_tile = ((enabled >> 5) & 3) == 1 ? 4 : (((enabled >> 5) & 3) == 2 ? 8 : 0);   // A/B measurements
  enabled &= 3;
  c->fast_mul = enabled < 0 ? 0 : (enabled > 2 ? 2 : enabled);
  return GTP_OK;
}

int gtp_from_host(gtp_ctx* c, int ndim, const uint64_t* shape, const uint64_t* degrees, const double* data, gtp_poly** out) {
  return wrap(c, [&] {
    GTP_CHECK(out && data && ndim >= 0 && ndim <= GTP_MAX_NDIM, GTP_ERR_ARG, "bad arguments");
    *out = from_values(*c, to_shape(shape, ndim), to_shape(degrees, ndim), data).release();
  });
}
int gtp_from_device(gtp_ctx* c, int ndim, const uint64_t* shape, const uint64_t* degrees, const double* dptr, gtp_poly** out) {
  return wrap(c, [&] {
    GTP_CHECK(out && dptr && ndim >= 0 && ndim <= GTP_MAX_NDIM, GTP_ERR_ARG, "bad arguments");
    auto b = std::make_shared<Buf>();
    b->d = const_cast<double*>(dptr);
    b->n = prod(to_shape(shape, ndim));
    b->owned = false;
    *out = make_poly(b, 0, to_shape(shape, ndim), to_shape(degrees, ndim)).release();
  });
}
int gtp_to_host(gtp_ctx* c, const gtp_poly* p, double* out) {
  return wrap(c, [&] {
    GTP_CHECK(p && out, GTP_ERR_ARG, "null argument");
    GTP_CUDA(cudaMemcpyAsync(out, p->ptr(), p->len() * sizeof(double), cudaMemcpyDefault, c->stream));   // scalar-pool slots are host memory
    c->sync();
  });
}
int gtp_device_ptr(gtp_ctx* c, const gtp_poly* p, const double** out) {
  return wrap(c, [&] {
    GTP_CHECK(p && out, GTP_ERR_ARG, "null argument");
    *out = p->ptr();
  });
}
int gtp_clone(gtp_ctx* c, const gtp_poly* p, gtp_poly** out) {
  return wrap(c, [&] {
    GTP_CHECK(p && out, GTP_ERR_ARG, "null argument");
    *out = share(*p).release();
  });
}
void gtp_free(gtp_ctx* c, gtp_poly* p) {
  if (c) cudaSetDevice(c->device);
  delete p;
}
int gtp_ndim(const gtp_poly* p) { return p->ndim(); }
uint64_t gtp_len(const gtp_poly* p) { return p->len(); }
void gtp_shape(const gtp_poly* p, uint64_t* out) { std::copy(p->shape.begin(), p->shape.end(), out); }
void gtp_degrees_p1(const gtp_poly* p, uint64_t* out) { std::copy(p->degrees.begin(), p->degrees.end(), out); }

int gtp_from_scalar(gtp_ctx* c, double x, gtp_poly** out) {
  return wrap(c, [&] { *out = scalar_poly(*c, x, {}, {}).release(); });
}
int gtp_zero_with(gtp_ctx* c, int ndim, const uint64_t* degrees, gtp_poly** out) {
  return wrap(c, [&] { *out = zero_with(*c, to_shape(degrees, ndim)).release(); });
}
static PolyP make_var(Ctx& c, u64 v, double x, u64 stored, bool one_coeff, Shape degrees) {
  Shape shape(degrees.size(), 1);
  shape[v] = stored;
  double vals[2] = {x, one_coeff ? 1.0 : 0.0};
  PolyP p;
  if (BufP slot = c.alloc_host_visible(vals, (int)stored)) p = make_poly(slot, 0, shape, degrees);
  else p = from_values(c, shape, degrees, vals);
  p->cls->known = true;
  p->cls->first = x;
  p->cls->linear = stored >= 2;  // [x, m] along v, every other entry absent
  p->cls->c = x;
  p->cls->m = vals[1];
  p->cls->v = v;
  return p;
}
int gtp_var(gtp_ctx* c, uint64_t v, double x, uint64_t len, gtp_poly** out) {  // :239-248
  return wrap(c, [&] {
    GTP_CHECK(v < (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "variable index too large");
    *out = make_var(*c, v, x, std::min<u64>(len, 2), len > 1, Shape(v + 1, len)).release();
  });
}
int gtp_var_at_zero(gtp_ctx* c, uint64_t v, uint64_t len, gtp_poly** out) {  // :228-237
  return wrap(c, [&] {
    GTP_CHECK(v < (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "variable index too large");
    *out = make_var(*c, v, 0.0, 2, len > 1, Shape(v + 1, len)).release();
  });
}
int gtp_var_with_degrees_p1(gtp_ctx* c, uint64_t v, double x, int ndim, const uint64_t* degrees, gtp_poly** out) {  // :250-259
  return wrap(c, [&] {
    GTP_CHECK((int)v < ndim, GTP_ERR_INDEX, "variable index out of range");
    *out = make_var(*c, v, x, 2, degrees[v] > 1, to_shape(degrees, ndim)).release();
  });
}

#define BINARY(name, expr)                                                                    \
  int name(gtp_ctx* c, const gtp_poly* a, const gtp_poly* b, gtp_poly** out) {                \
    return wrap(c, [&] {                                                                      \
      GTP_CHECK(a && b && out, GTP_ERR_ARG, "null argument");                                 \
      *out = (expr).release();                                                                \
    });                                                                                       \
  }
BINARY(gtp_add, poly_add(*c, *a, *b, false))
BINARY(gtp_sub, poly_add(*c, *a, *b, true))
BINARY(gtp_mul, poly_mul(*c, *a, *b))
BINARY(gtp_div, poly_div(*c, *a, *b))
#undef BINARY

int gtp_neg(gtp_ctx* c, const gtp_poly* a, gtp_poly** out) { return wrap(c, [&] { *out = poly_neg(*c, *a).release(); }); }
int gtp_exp(gtp_ctx* c, const gtp_poly* a, gtp_poly** out) { return wrap(c, [&] { *out = poly_exp_log(*c, *a, false).release(); }); }
int gtp_log(gtp_ctx* c, const gtp_poly* a, gtp_poly** out) { return wrap(c, [&] { *out = poly_exp_log(*c, *a, true).release(); }); }
int gtp_pow(gtp_ctx* c, const gtp_poly* a, uint32_t e, gtp_poly** out) { return wrap(c, [&] { *out = poly_pow(*c, *a, e).release(); }); }

int gtp_derivative(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out) {  // :457-481
  return wrap(c, [&] {
    GTP_CHECK(v < a->degrees.size() && n < a->degrees[v], GTP_ERR_INDEX, "derivative: variable / order out of range");
    *out = slice_scale(*c, *a, v, n, 0).release();
  });
}
int gtp_taylor_expansion_of_coeff(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out) {  // :484-509
  return wrap(c, [&] { *out = slice_scale(*c, *a, v, n, 1).release(); });
}
int gtp_shift_down(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t n, gtp_poly** out) {
  return wrap(c, [&] { *out = poly_shift_down(*c, *a, v, n).release(); });
}
int gtp_coefficients_of_term(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t order, gtp_poly** out) {  // :341-358
  return wrap(c, [&] {
    if (v >= a->shape.size()) {
      *out = (order == 0 ? share(*a) : zero_with(*c, a->degrees)).release();
      return;
    }
    if (order >= a->shape[v]) {
      *out = zero_with(*c, a->degrees).release();
      return;
    }
    Shape ext = a->shape, lo(a->shape.size(), 0);
    ext[v] = 1;
    lo[v] = order;
    *out = copy_box(*c, *a, lo, ext, a->degrees).release();
  });
}
int gtp_taylor_polynomial(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t order, gtp_poly** out) {  // :360-378
  return wrap(c, [&] {
    GTP_CHECK(v < a->degrees.size() && order < a->degrees[v], GTP_ERR_INDEX, "taylor_polynomial: variable / order out of range");
    if (order >= a->shape[v]) {
      *out = share(*a).release();
      return;
    }
    Shape ext = a->shape;
    ext[v] = std::min(a->shape[v], order + 1);
    *out = copy_box(*c, *a, Shape(ext.size(), 0), ext, a->degrees).release();
  });
}
int gtp_taylor_polynomial_terms(gtp_ctx* c, const gtp_poly* a, uint64_t v, const uint64_t* orders, int n_orders, gtp_poly** out) {  // :380-404
  return wrap(c, [&] {
    u64 max_order_p1 = 1;
    bool has0 = false;
    for (int i = 0; i < n_orders; i++) {
      max_order_p1 = std::max(max_order_p1, orders[i] + 1);
      has0 |= orders[i] == 0;
    }
    if (v >= a->shape.size()) {
      *out = (has0 ? share(*a) : zero_with(*c, a->degrees)).release();
      return;
    }
    u64 upper = std::min(a->shape[v], max_order_p1);
    std::vector<unsigned char> keep(max_order_p1, 0);
    for (int i = 0; i < n_orders; i++) keep[orders[i]] = 1;
    // the keep mask is integer metadata: staged through a small device byte array
    BufP kb = c->alloc((max_order_p1 + 7) / 8 + 1);
    GTP_CUDA(cudaMemcpyAsync(kb->d, keep.data(), max_order_p1, cudaMemcpyHostToDevice, c->stream));
    c->sync();
    Shape ext = a->shape;
    ext[v] = upper;
    PolyP r = new_uninit(*c, ext, a->degrees);
    EwOperand A;
    A.p = a->ptr();
    A.shape = a->shape;
    launch_ew(*c, EW_MASK, ext, A, nullptr, r->buf->d, ext, {}, (int)v, nullptr, (const unsigned char*)kb->d);
    *out = r.release();
  });
}
int gtp_subst_var(gtp_ctx* c, const gtp_poly* a, uint64_t v, const gtp_poly* s, gtp_poly** out) {
  return wrap(c, [&] { *out = poly_subst_var(*c, *a, v, *s).release(); });
}
int gtp_truncate_to_degree_p1(gtp_ctx* c, const gtp_poly* a, uint64_t d, gtp_poly** out) {  // :183-193
  return wrap(c, [&] { *out = truncate_degrees(*c, *a, Shape(a->degrees.size(), d)).release(); });
}
int gtp_remove_last_variable(gtp_ctx* c, const gtp_poly* a, gtp_poly** out) {  // :172-181
  return wrap(c, [&] {
    GTP_CHECK(!a->degrees.empty(), GTP_ERR_INDEX, "remove_last_variable on a 0-variable polynomial");
    size_t v = a->degrees.size() - 1;
    Shape d(a->degrees.begin(), a->degrees.end() - 1);
    Shape s(a->shape.begin(), a->shape.end() - 1);
    if (a->shape[v] == 1) {
      *out = make_poly(buf_of(*a), a->off, s, d).release();
      return;
    }
    Shape ext = a->shape;
    ext[v] = 1;
    PolyP r = copy_box(*c, *a, Shape(ext.size(), 0), ext, a->degrees);
    *out = make_poly(r->buf, 0, s, d).release();
  });
}
int gtp_extend_to_dim(gtp_ctx* c, const gtp_poly* a, uint64_t ndim, uint64_t degree_p1, gtp_poly** out) {  // :81-89
  return wrap(c, [&] {
    GTP_CHECK(a->shape.size() <= ndim && ndim <= (u64)GTP_MAX_NDIM, GTP_ERR_ARG, "extend_to_dim: bad ndim");
    PolyP r = share(*a);
    r->shape.resize(ndim, 1);
    r->degrees.resize(ndim, degree_p1);
    check_invariants(r->shape, r->degrees);
    *out = r.release();
  });
}
int gtp_extend(gtp_ctx* c, const gtp_poly* a, int ndim, const uint64_t* new_size, gtp_poly** out) {  // :91-112
  return wrap(c, [&] {
    Shape ns = to_shape(new_size, ndim);
    GTP_CHECK(a->shape.size() <= ns.size(), GTP_ERR_ARG, "extend: fewer axes than the source");
    Shape src = a->shape;
    src.resize(ns.size(), 1);
    for (size_t i = 0; i < ns.size(); i++) GTP_CHECK(src[i] <= ns[i], GTP_ERR_SHAPE, "extend: new size smaller than stored shape");
    PolyP r = new_zeros(*c, ns, ns);
    EwOperand A;
    A.p = a->ptr();
    A.shape = src;
    launch_ew(*c, EW_COPY, src, A, nullptr, r->buf->d, ns, {});
    *out = r.release();
  });
}

int gtp_constant_term(gtp_ctx* c, const gtp_poly* a, double* out) {  // :296-299
  return wrap(c, [&] {
    if (a->len() <= 8192) {   // small: classification (cached per handle) already carries coeffs.first()
      classify(*c, *a);
      *out = a->cls->first;
      return;
    }
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], a->ptr(), sizeof(double), cudaMemcpyDefault, c->stream));
    c->sync();
    *out = c->rb_host->vals[0];
  });
}
int gtp_coefficient(gtp_ctx* c, const gtp_poly* a, const uint64_t* index, int n_index, double* out) {  // :314-339
  return wrap(c, [&] {
    u64 off = 0;
    for (int v = 0; v < n_index; v++) {
      u64 len_of = (size_t)v < a->degrees.size() ? a->degrees[v] : UNB;
      GTP_CHECK(index[v] < len_of, GTP_ERR_INDEX, "index out of bounds");
      if ((size_t)v >= a->shape.size()) {
        if (index[v] != 0) { *out = 0.0; return; }
      } else if (index[v] >= a->shape[v]) {
        *out = 0.0;
        return;
      } else {
        off += index[v] * stride_of(a->shape, v);
      }
    }
    GTP_CHECK((size_t)n_index >= a->shape.size(), GTP_ERR_INDEX, "index is too short");
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], a->ptr() + off, sizeof(double), cudaMemcpyDefault, c->stream));
    c->sync();
    *out = c->rb_host->vals[0];
  });
}
int gtp_gather_axis(gtp_ctx* c, const gtp_poly* a, uint64_t v, uint64_t count, double* out) {
  return wrap(c, [&] {
    GTP_CHECK(out, GTP_ERR_ARG, "null argument");
    if (count == 0) return;
    u64 len = v < a->shape.size() ? a->shape[v] : 1;
    u64 stride = v < a->shape.size() ? stride_of(a->shape, v) : 0;
    BufP tmp = c->alloc(count);
    launch_gather_strided(*c, a->ptr(), stride, len, count, tmp->d);
    GTP_CUDA(cudaMemcpyAsync(c->host_staging(count), tmp->d, count * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
    std::memcpy(out, c->gather_host, count * sizeof(double));
  });
}
int gtp_extract_constant(gtp_ctx* c, const gtp_poly* a, int* is_constant, double* value) {  // :262-269
  return wrap(c, [&] {
    *is_constant = a->len() == 1;
    if (*is_constant) {
      classify(*c, *a);
      *value = a->cls->first;
    }
  });
}
int gtp_extract_linear(gtp_ctx* c, const gtp_poly* a, int* is_linear, double* cst, double* m, uint64_t* v) {  // :275-294
  return wrap(c, [&] {
    *is_linear = 0;
    if (a->len() == 1) return;  // constants are not recognised
    classify(*c, *a);
    if (a->cls->linear) {
      *is_linear = 1;
      *cst = a->cls->c;
      *m = a->cls->m;
      *v = a->cls->v;
    }
  });
}
int gtp_is_zero(gtp_ctx* c, const gtp_poly* a, int* out) { return wrap(c, [&] { *out = is_zero(*c, *a); }); }
int gtp_is_one(gtp_ctx* c, const gtp_poly* a, int* out) { return wrap(c, [&] { *out = is_one(*c, *a); }); }
int gtp_evaluate_all_one(gtp_ctx* c, const gtp_poly* a, double* out) {  // :583-586
  return wrap(c, [&] {
    launch_sum_all(*c, a->ptr(), a->len(), &c->rb_dev->vals[0]);
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], &c->rb_dev->vals[0], sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
    *out = c->rb_host->vals[0];
  });
}
int gtp_eq(gtp_ctx* c, const gtp_poly* a, const gtp_poly* b, int* out) {
  return wrap(c, [&] {
    *out = 0;
    if (a->shape != b->shape || a->degrees != b->degrees) return;
    launch_eq(*c, a->ptr(), b->ptr(), a->len(), c->rb_dev);
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->flag, &c->rb_dev->flag, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
    *out = c->rb_host->flag ? 1 : 0;
  });
}

int gtp_mul_rows_raw(gtp_ctx* c, int ndim, const uint64_t* xshape, const double* x, const uint64_t* yshape, const double* y,
                     const uint64_t* rshape, uint64_t row_begin, uint64_t row_step, uint64_t row_count, double* out_rows) {
  return wrap(c, [&] {
    GTP_CHECK(ndim >= 1 && ndim <= GTP_MAX_NDIM && x && y && out_rows, GTP_ERR_ARG, "bad arguments");
    MulArgs m;
    m.ndim = ndim;
    m.xs = to_shape(xshape, ndim);
    m.ys = to_shape(yshape, ndim);
    m.rs = to_shape(rshape, ndim);
    GTP_CHECK(row_step >= 1 && (row_count == 0 || row_begin + (row_count - 1) * row_step < m.rs[0]), GTP_ERR_INDEX,
              "row range outside the result's leading axis");
    m.x = x;
    m.y = y;
    m.out = out_rows;
    m.row_begin = row_begin;
    m.row_step = row_step;
    m.row_count = row_count;
    launch_mul(*c, m);
  });
}
int gtp_mul_rowlist_raw(gtp_ctx* c, int ndim, const uint64_t* xshape, const double* x, const uint64_t* yshape, const double* y,
                        const uint64_t* rshape, const uint64_t* rows, uint64_t n_rows, double* out_rows) {
  return wrap(c, [&] {
    GTP_CHECK(ndim >= 1 && ndim <= GTP_MAX_NDIM && x && y && out_rows && (rows || n_rows == 0), GTP_ERR_ARG, "bad arguments");
    MulArgs m;
    m.ndim = ndim;
    m.xs = to_shape(xshape, ndim);
    m.ys = to_shape(yshape, ndim);
    m.rs = to_shape(rshape, ndim);
    if (n_rows == 0) return;
    for (uint64_t i = 0; i < n_rows; i++)
      GTP_CHECK(rows[i] < m.rs[0], GTP_ERR_INDEX, "row outside the result's leading axis");
    m.x = x;
    m.y = y;
    m.out = out_rows;
    m.rows.assign(rows, rows + n_rows);
    launch_mul(*c, m);
  });
}
double gtp_mul_macs(int ndim, const uint64_t* xs, const uint64_t* ys, const uint64_t* rs) {
  return mul_macs(to_shape(xs, ndim), to_shape(ys, ndim), to_shape(rs, ndim));
}
int gtp_mul_kernel_kind(gtp_ctx* c, int ndim, const uint64_t* xs, const uint64_t* ys, const uint64_t* rs) {
  MulArgs m;
  m.ndim = ndim;
  m.xs = to_shape(xs, ndim);
  m.ys = to_shape(ys, ndim);
  m.rs = to_shape(rs, ndim);
  m.row_count = m.rs.empty() ? 1 : m.rs[0];
  int kind = 0;
  wrap(c, [&] { kind = mul_kernel_kind(*c, m); });   // planning queries the device (cooperative-kernel occupancy)
  return kind;
}
int gtp_fp64_peak_probe(gtp_ctx* c, int kind, int iters, double* flops, double* ms) {
  return wrap(c, [&] { fp64_peak_probe(*c, kind, iters, flops, ms); });
}

}  // extern "C"
