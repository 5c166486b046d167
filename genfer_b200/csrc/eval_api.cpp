// C ABI of the host evaluator (SURVEY 8 f1): runs an SGCL program end to end -- parse, translate to a
// generating function, simplify, evaluate moments and probabilities -- with EVERY Taylor-polynomial operation
// going through the C ABI of libgenfer_taylor (gtp_*, i.e. the CUDA kernels).  It plays the role of the
// reference's `run()` / `run_program::<F64>` (src/main.rs:108-227) with GenFun::eval (src/generating_function.rs)
// as the caller of TaylorPoly.  Host logic only; there is no CPU arithmetic path here: without a CUDA context
// the calls fail.
#include <cstring>
#include <memory>

#include "../../include/genfer_taylor.h"
#include "evaluator/report.hpp"
#include "interval.cuh"

namespace {

struct GpuBackend {
  gtp_ctx* ctx;
  struct Handle {
    gtp_ctx* c;
    gtp_poly* p;
    Handle(gtp_ctx* c_, gtp_poly* p_) : c(c_), p(p_) {}
    ~Handle() { if (p) gtp_free(c, p); }
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
  };
  using Poly = std::shared_ptr<Handle>;
  using Scalar = double;   // the f64 Number path (the only one on the device)
  static double scalar_max(double x, double y) { return x > y ? x : y; }   // F64::max (number/f64.rs:77-84)

  void check(int rc) const {
    if (rc != 0) throw gfe::EvalError(std::string("libgenfer_taylor: ") + gtp_last_error(ctx));
  }
  Poly wrap(gtp_poly* p) const { return std::make_shared<Handle>(ctx, p); }
  static std::vector<uint64_t> u64(const std::vector<size_t>& v) { return std::vector<uint64_t>(v.begin(), v.end()); }

  Poly from_scalar(double x) { gtp_poly* o; check(gtp_from_scalar(ctx, x, &o)); return wrap(o); }
  Poly var(gfe::Var v, double x, size_t len) { gtp_poly* o; check(gtp_var(ctx, v, x, len, &o)); return wrap(o); }
  Poly var_at_zero(gfe::Var v, size_t len) { gtp_poly* o; check(gtp_var_at_zero(ctx, v, len, &o)); return wrap(o); }
  Poly var_with_degrees(gfe::Var v, double x, const std::vector<uint64_t>& d) {
    gtp_poly* o; check(gtp_var_with_degrees_p1(ctx, v, x, (int)d.size(), d.data(), &o)); return wrap(o);
  }
  Poly zero_with(const std::vector<uint64_t>& d) { gtp_poly* o; check(gtp_zero_with(ctx, (int)d.size(), d.data(), &o)); return wrap(o); }
  Poly new_poly(const std::vector<uint64_t>& shape, const std::vector<uint64_t>& degrees, const double* data) {
    gtp_poly* o; check(gtp_from_host(ctx, (int)shape.size(), shape.data(), degrees.data(), data, &o)); return wrap(o);
  }
#define GFE_BIN(name, fn) Poly name(const Poly& a, const Poly& b) { gtp_poly* o; check(fn(ctx, a->p, b->p, &o)); return wrap(o); }
  GFE_BIN(add, gtp_add) GFE_BIN(sub, gtp_sub) GFE_BIN(mul, gtp_mul) GFE_BIN(div, gtp_div)
#undef GFE_BIN
  Poly neg(const Poly& a) { gtp_poly* o; check(gtp_neg(ctx, a->p, &o)); return wrap(o); }
  Poly exp(const Poly& a) { gtp_poly* o; check(gtp_exp(ctx, a->p, &o)); return wrap(o); }
  Poly log(const Poly& a) { gtp_poly* o; check(gtp_log(ctx, a->p, &o)); return wrap(o); }
  Poly pow(const Poly& a, uint32_t e) { gtp_poly* o; check(gtp_pow(ctx, a->p, e, &o)); return wrap(o); }
  Poly derivative(const Poly& a, gfe::Var v, size_t n) { gtp_poly* o; check(gtp_derivative(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly taylor_expansion_of_coeff(const Poly& a, gfe::Var v, size_t n) { gtp_poly* o; check(gtp_taylor_expansion_of_coeff(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly shift_down(const Poly& a, gfe::Var v, size_t n) { gtp_poly* o; check(gtp_shift_down(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly coefficients_of_term(const Poly& a, gfe::Var v, size_t n) { gtp_poly* o; check(gtp_coefficients_of_term(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly taylor_polynomial_terms(const Poly& a, gfe::Var v, const std::vector<size_t>& orders) {
    std::vector<uint64_t> os = u64(orders);
    gtp_poly* o; check(gtp_taylor_polynomial_terms(ctx, a->p, v, os.data(), (int)os.size(), &o)); return wrap(o);
  }
  Poly subst_var(const Poly& a, gfe::Var v, const Poly& s) { gtp_poly* o; check(gtp_subst_var(ctx, a->p, v, s->p, &o)); return wrap(o); }
  Poly truncate_to_degree_p1(const Poly& a, size_t d) { gtp_poly* o; check(gtp_truncate_to_degree_p1(ctx, a->p, d, &o)); return wrap(o); }
  Poly remove_last_variable(const Poly& a) { gtp_poly* o; check(gtp_remove_last_variable(ctx, a->p, &o)); return wrap(o); }
  Poly extend_to_dim(const Poly& a, size_t ndim, size_t d) { gtp_poly* o; check(gtp_extend_to_dim(ctx, a->p, ndim, d, &o)); return wrap(o); }
  double constant_term(const Poly& a) { double x; check(gtp_constant_term(ctx, a->p, &x)); return x; }
  std::vector<double> gather_axis(const Poly& a, gfe::Var v, size_t count) {
    std::vector<double> out(count);
    if (count) check(gtp_gather_axis(ctx, a->p, v, count, out.data()));
    return out;
  }
  size_t num_vars(const Poly& a) { return (size_t)gtp_ndim(a->p); }
  std::vector<uint64_t> array_shape(const Poly& a) {
    std::vector<uint64_t> s((size_t)gtp_ndim(a->p) + 1);
    gtp_shape(a->p, s.data());
    s.resize((size_t)gtp_ndim(a->p));
    return s;
  }
  std::optional<double> extract_constant(const Poly& a) {
    int is_c = 0; double v = 0;
    check(gtp_extract_constant(ctx, a->p, &is_c, &v));
    if (is_c) return v;
    return std::nullopt;
  }
  std::vector<double> to_host(const Poly& a) {
    std::vector<double> out(gtp_len(a->p));
    check(gtp_to_host(ctx, a->p, out.data()));
    return out;
  }

  // ---- TaylorExpansion<F64> (univariate_taylor.rs) for the symbolic mode: a gtu_program per evaluation -----------------
  // Every operator records into the current program; the variant and order of each value are known on the host at once.
  // The first coefficient read of an evaluation runs the program (one launch, one read-back of the whole value); further
  // reads of that value come from the host copy.  The next value recorded after a run starts a new program.
  struct Program {
    gtp_ctx* c;
    gtu_program* p;
    bool ran = false;
    uint32_t read_slot = 0;     // the value whose coefficients `host` holds (valid once ran)
    std::vector<double> host;
    Program(gtp_ctx* c_, gtu_program* p_) : c(c_), p(p_) {}
    ~Program() { gtu_program_free(c, p); }
    Program(const Program&) = delete;
    Program& operator=(const Program&) = delete;
  };
  struct Uni {
    std::shared_ptr<Program> prog;
    uint32_t slot = 0;
    bool is_const = true;
    uint64_t n = 1;
  };
  std::shared_ptr<Program> cur;
  gtu_program* recording() {
    if (!cur || cur->ran) {
      gtu_program* p;
      check(gtu_program_create(ctx, &p));
      cur = std::make_shared<Program>(ctx, p);
    }
    return cur->p;
  }
  Uni uni_slot(uint32_t slot) {
    Uni u{cur, slot, true, 1};
    int is_c = 0;
    check(gtu_program_slot(cur->p, slot, &is_c, &u.n));
    u.is_const = is_c != 0;
    if (u.is_const) u.n = 1;
    return u;
  }
  Uni uni_op(int op, const Uni& a, const Uni* b, uint32_t e = 0) {
    gtu_program* p = recording();
    if (a.prog != cur || (b && b->prog != cur)) throw gfe::EvalError("univariate value used after its program ran");
    uint32_t s;
    check(gtu_program_op(ctx, p, op, a.slot, b ? b->slot : 0, e, &s));
    return uni_slot(s);
  }
  Uni uni_constant(double x) { uint32_t s; check(gtu_program_constant(ctx, recording(), x, &s)); return uni_slot(s); }
  Uni uni_var(double x, size_t order) { uint32_t s; check(gtu_program_var(ctx, recording(), x, order, &s)); return uni_slot(s); }
  Uni uni_add(const Uni& a, const Uni& b) { return uni_op(GTU_ADD, a, &b); }
  Uni uni_mul(const Uni& a, const Uni& b) { return uni_op(GTU_MUL, a, &b); }
  Uni uni_div(const Uni& a, const Uni& b) { return uni_op(GTU_DIV, a, &b); }
  Uni uni_exp(const Uni& a) { return uni_op(GTU_EXP, a, nullptr); }
  Uni uni_log(const Uni& a) { return uni_op(GTU_LOG, a, nullptr); }
  Uni uni_pow(const Uni& a, uint32_t e) { return uni_op(GTU_POW, a, nullptr, e); }
  Uni uni_max(const Uni& a, const Uni& b) {   // :219-224: constants only
    if (!a.is_const || !b.is_const) throw gfe::EvalError("Maximum can only be applied to constant Taylor expansions.");
    return uni_op(GTU_MAX, a, &b);
  }
  double uni_coeff(const Uni& a, size_t order) {   // gtu_coeff (:25-36) of the value
    if (a.is_const && order != 0) return 0.0;
    if (!a.is_const && order >= a.n) throw gfe::EvalError("libgenfer_taylor: coeff: index out of bounds");
    Program& pr = *a.prog;
    if (!pr.ran || pr.read_slot != a.slot) {
      pr.host.resize(a.n);
      check(gtu_program_run(ctx, pr.p, &a.slot, 1, pr.host.data()));
      pr.ran = true;
      pr.read_slot = a.slot;
    }
    return pr.host[a.is_const ? 0 : order];
  }
};

// Interval<F64> as the evaluator sees it (src/interval.rs): constructible from an f64 constant (a point interval); the
// arithmetic is interval.cuh's, the same functions the kernels run.
struct IvS {
  gti::Iv v{0.0, 0.0};
  IvS() = default;
  IvS(double x) : v{x, x} {}
  explicit IvS(gti::Iv i) : v(i) {}
  static IvS from_bounds(double lo, double hi) { return IvS(gti::iv(lo, hi)); }
  double lower() const { return v.lo; }
  double upper() const { return v.hi; }
  friend IvS operator+(const IvS& a, const IvS& b) { return IvS(gti::iv_add(a.v, b.v)); }
  friend IvS operator-(const IvS& a, const IvS& b) { return IvS(gti::iv_sub(a.v, b.v)); }
  friend IvS operator*(const IvS& a, const IvS& b) { return IvS(gti::iv_mul(a.v, b.v)); }
  friend IvS operator/(const IvS& a, const IvS& b) { return IvS(gti::iv_div(a.v, b.v)); }
  friend bool operator==(const IvS& a, const IvS& b) { return a.v.lo == b.v.lo && a.v.hi == b.v.hi; }
};

// TaylorPoly<Interval<F64>> on the device (gti_*, interval_api.cu): the number type of the reference's --bounds mode
struct GpuIvBackend {
  gtp_ctx* ctx;
  struct Handle {
    gtp_ctx* c;
    gti_poly* p;
    Handle(gtp_ctx* c_, gti_poly* p_) : c(c_), p(p_) {}
    ~Handle() { if (p) gti_free(c, p); }
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
  };
  using Poly = std::shared_ptr<Handle>;
  using Scalar = IvS;
  static IvS scalar_max(const IvS& x, const IvS& y) {   // Interval::max: componentwise
    return IvS(gti::iv(x.v.lo > y.v.lo ? x.v.lo : y.v.lo, x.v.hi > y.v.hi ? x.v.hi : y.v.hi));
  }
  void check(int rc) const {
    if (rc != 0) throw gfe::EvalError(std::string("libgenfer_taylor: ") + gtp_last_error(ctx));
  }
  Poly wrap(gti_poly* p) const { return std::make_shared<Handle>(ctx, p); }

  Poly from_scalar(const IvS& x) { gti_poly* o; check(gti_from_scalar(ctx, x.v.lo, x.v.hi, &o)); return wrap(o); }
  Poly var(gfe::Var v, const IvS& x, size_t len) { gti_poly* o; check(gti_var(ctx, v, x.v.lo, x.v.hi, len, &o)); return wrap(o); }
  Poly var_at_zero(gfe::Var v, size_t len) { gti_poly* o; check(gti_var_at_zero(ctx, v, len, &o)); return wrap(o); }
  Poly var_with_degrees(gfe::Var v, const IvS& x, const std::vector<uint64_t>& d) {
    gti_poly* o; check(gti_var_with_degrees_p1(ctx, v, x.v.lo, x.v.hi, (int)d.size(), d.data(), &o)); return wrap(o);
  }
  Poly zero_with(const std::vector<uint64_t>& d) { gti_poly* o; check(gti_zero_with(ctx, (int)d.size(), d.data(), &o)); return wrap(o); }
  Poly new_poly(const std::vector<uint64_t>& shape, const std::vector<uint64_t>& degrees, const double* data) {   // f64 GenFun constants
    gti_poly* o; check(gti_from_host(ctx, (int)shape.size(), shape.data(), degrees.data(), data, 0, &o)); return wrap(o);
  }
  Poly new_poly(const std::vector<uint64_t>& shape, const std::vector<uint64_t>& degrees, const IvS* data) {
    static_assert(sizeof(IvS) == 2 * sizeof(double), "IvS is a (lo, hi) pair");
    gti_poly* o; check(gti_from_host(ctx, (int)shape.size(), shape.data(), degrees.data(), reinterpret_cast<const double*>(data), 1, &o)); return wrap(o);
  }
#define GFE_BIN(name, fn) Poly name(const Poly& a, const Poly& b) { gti_poly* o; check(fn(ctx, a->p, b->p, &o)); return wrap(o); }
  GFE_BIN(add, gti_add) GFE_BIN(sub, gti_sub) GFE_BIN(mul, gti_mul) GFE_BIN(div, gti_div)
#undef GFE_BIN
  Poly neg(const Poly& a) { gti_poly* o; check(gti_neg(ctx, a->p, &o)); return wrap(o); }
  Poly exp(const Poly& a) { gti_poly* o; check(gti_exp(ctx, a->p, &o)); return wrap(o); }
  Poly log(const Poly& a) { gti_poly* o; check(gti_log(ctx, a->p, &o)); return wrap(o); }
  Poly pow(const Poly& a, uint32_t e) { gti_poly* o; check(gti_pow(ctx, a->p, e, &o)); return wrap(o); }
  Poly derivative(const Poly& a, gfe::Var v, size_t n) { gti_poly* o; check(gti_derivative(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly taylor_expansion_of_coeff(const Poly& a, gfe::Var v, size_t n) { gti_poly* o; check(gti_taylor_expansion_of_coeff(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly shift_down(const Poly& a, gfe::Var v, size_t n) { gti_poly* o; check(gti_shift_down(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly coefficients_of_term(const Poly& a, gfe::Var v, size_t n) { gti_poly* o; check(gti_coefficients_of_term(ctx, a->p, v, n, &o)); return wrap(o); }
  Poly taylor_polynomial_terms(const Poly& a, gfe::Var v, const std::vector<size_t>& orders) {
    std::vector<uint64_t> os(orders.begin(), orders.end());
    gti_poly* o; check(gti_taylor_polynomial_terms(ctx, a->p, v, os.data(), (int)os.size(), &o)); return wrap(o);
  }
  Poly subst_var(const Poly& a, gfe::Var v, const Poly& s) { gti_poly* o; check(gti_subst_var(ctx, a->p, v, s->p, &o)); return wrap(o); }
  Poly truncate_to_degree_p1(const Poly& a, size_t d) { gti_poly* o; check(gti_truncate_to_degree_p1(ctx, a->p, d, &o)); return wrap(o); }
  Poly remove_last_variable(const Poly& a) { gti_poly* o; check(gti_remove_last_variable(ctx, a->p, &o)); return wrap(o); }
  Poly extend_to_dim(const Poly& a, size_t ndim, size_t d) { gti_poly* o; check(gti_extend_to_dim(ctx, a->p, ndim, d, &o)); return wrap(o); }
  IvS constant_term(const Poly& a) { double x[2]; check(gti_constant_term(ctx, a->p, x)); return IvS(gti::iv(x[0], x[1])); }
  std::vector<IvS> gather_axis(const Poly& a, gfe::Var v, size_t count) {
    std::vector<IvS> out(count);
    if (count) check(gti_gather_axis(ctx, a->p, v, count, reinterpret_cast<double*>(out.data())));
    return out;
  }
  size_t num_vars(const Poly& a) { return (size_t)gti_ndim(a->p); }
  std::vector<uint64_t> array_shape(const Poly& a) {
    std::vector<uint64_t> s((size_t)gti_ndim(a->p) + 1);
    gti_shape(a->p, s.data());
    s.resize((size_t)gti_ndim(a->p));
    return s;
  }
  std::optional<IvS> extract_constant(const Poly& a) {
    int is_c = 0; double v[2] = {0, 0};
    check(gti_extract_constant(ctx, a->p, &is_c, v));
    if (is_c) return IvS(gti::iv(v[0], v[1]));
    return std::nullopt;
  }
  std::vector<IvS> to_host(const Poly& a) {
    std::vector<IvS> out(gti_len(a->p));
    check(gti_to_host(ctx, a->p, reinterpret_cast<double*>(out.data())));
    return out;
  }
};

}  // namespace

struct gtp_sgcl_result {
  gfe::RunResult r;
};

extern "C" {

int gtp_run_sgcl(gtp_ctx* ctx, const char* source, int64_t limit, int flags, uint64_t unroll, gtp_sgcl_result** out,
                 char* err, size_t err_cap) {
  if (!ctx || !source || !out) return GTP_ERR_ARG;
  try {
    gfe::RunOptions opt;
    if (limit >= 0) opt.limit = (size_t)limit;
    opt.no_probs = (flags & 1) != 0;
    opt.no_simplify_gf = (flags & 2) != 0;
    opt.bounds = (flags & 4) != 0;
    opt.symbolic = (flags & 8) != 0;
    opt.unroll = (size_t)unroll;
    auto res = std::make_unique<gtp_sgcl_result>();
    if (opt.bounds) {   // --bounds: run_program_intervals::<F64> (main.rs:145-185) over TaylorPoly<Interval<F64>> on the device
      GpuIvBackend backend{ctx};
      res->r = gfe::run_program(backend, source, opt);
    } else {
      GpuBackend backend{ctx};
      res->r = gfe::run_program(backend, source, opt);
    }
    *out = res.release();
    return GTP_OK;
  } catch (const std::exception& e) {
    if (err && err_cap) {
      std::strncpy(err, e.what(), err_cap - 1);
      err[err_cap - 1] = '\0';
    }
    return GTP_ERR_INDEX;   // the reference panics on every error of this path (parse error, assert!)
  }
}
// The --bounds-style enclosure of the evaluator's direct outputs with the interval arithmetic on the device (SURVEY 8 f3): the
// same host logic over TaylorPoly<Interval<F64>> (gti_*).  GenFun constants are the f64 values of the f64 path, as point
// intervals; no simplification pass (its polynomial form stores f64 coefficients).  Constants that come from a ratio in the
// program text are the enclosures Number::from_ratio builds (evaluator/num.hpp), so the result encloses the exact posterior.
// out12: [rest lo, hi, total lo, hi, raw moment 1..4 lo, hi]; probs_lohi: `limit` (lo, hi) pairs (may be null when limit <= 0).
int gtp_run_sgcl_bounds(gtp_ctx* ctx, const char* source, int64_t limit, uint64_t unroll, double* out12, double* probs_lohi,
                        char* err, size_t err_cap) {
  if (!ctx || !source || !out12) return GTP_ERR_ARG;
  try {
    GpuIvBackend backend{ctx};
    gfe::Program program = gfe::parse_program(source);
    gfe::GfTransformer transformer((size_t)unroll);
    gfe::GfTranslation tr = transformer.semantics(program);
    gfe::Evaluator<GpuIvBackend> ev(backend);
    IvS rest = backend.constant_term(ev.eval(tr.rest, std::vector<IvS>(tr.var_info.num_vars(), IvS(0.0)), 1));
    auto mom = ev.moments_taylor(tr.gf, program.result, tr.var_info, 5);
    out12[0] = rest.v.lo; out12[1] = rest.v.hi;
    out12[2] = mom.first.v.lo; out12[3] = mom.first.v.hi;
    for (size_t i = 0; i < 4; i++) { out12[4 + 2 * i] = mom.second.at(i).v.lo; out12[5 + 2 * i] = mom.second.at(i).v.hi; }
    if (limit > 0 && probs_lohi) {
      std::vector<IvS> p = ev.probs_taylor(tr.gf, program.result, tr.var_info, (size_t)limit);
      for (size_t i = 0; i < (size_t)limit; i++) { probs_lohi[2 * i] = p.at(i).v.lo; probs_lohi[2 * i + 1] = p.at(i).v.hi; }
    }
    return GTP_OK;
  } catch (const std::exception& e) {
    if (err && err_cap) {
      std::strncpy(err, e.what(), err_cap - 1);
      err[err_cap - 1] = '\0';
    }
    return GTP_ERR_INDEX;
  }
}
void gtp_sgcl_free(gtp_sgcl_result* r) { delete r; }
const char* gtp_sgcl_report(const gtp_sgcl_result* r) { return r->r.report.c_str(); }
void gtp_sgcl_moments(const gtp_sgcl_result* r, double* out11) {
  const gfe::RunResult& x = r->r;
  const double v[11] = {x.total, x.mean, x.raw2, x.raw3, x.raw4, x.stddev, x.variance, x.central3, x.central4, x.skewness, x.kurtosis};
  std::memcpy(out11, v, sizeof(v));
}
uint64_t gtp_sgcl_limit(const gtp_sgcl_result* r) { return r->r.probs.size(); }
int gtp_sgcl_is_normalized(const gtp_sgcl_result* r) { return r->r.is_normalized ? 1 : 0; }
void gtp_sgcl_probs(const gtp_sgcl_result* r, double* unnormalized, double* normalized) {
  const gfe::RunResult& x = r->r;
  for (size_t i = 0; i < x.probs.size(); i++) {
    if (unnormalized) unnormalized[i] = x.probs[i];
    if (normalized) normalized[i] = x.is_normalized ? x.probs[i] : x.normalized_probs[i];
  }
}
void gtp_sgcl_moment_bounds(const gtp_sgcl_result* r, double* out22) {
  for (size_t i = 0; i < r->r.moment_bounds.size() && i < 11; i++) {
    out22[2 * i] = r->r.moment_bounds[i].lo;
    out22[2 * i + 1] = r->r.moment_bounds[i].hi;
  }
}
void gtp_sgcl_prob_bounds(const gtp_sgcl_result* r, double* unnormalized_pairs, double* normalized_pairs) {
  const gfe::RunResult& x = r->r;
  for (size_t i = 0; i < x.prob_bounds.size(); i++) {
    const gfe::Iv n = x.is_normalized ? x.prob_bounds[i] : x.normalized_prob_bounds[i];
    if (unnormalized_pairs) { unnormalized_pairs[2 * i] = x.prob_bounds[i].lo; unnormalized_pairs[2 * i + 1] = x.prob_bounds[i].hi; }
    if (normalized_pairs) { normalized_pairs[2 * i] = n.lo; normalized_pairs[2 * i + 1] = n.hi; }
  }
}
void gtp_sgcl_stats(const gtp_sgcl_result* r, uint64_t* nodes_evaluated, uint64_t* cache_hits) {
  if (nodes_evaluated) *nodes_evaluated = r->r.nodes_evaluated;
  if (cache_hits) *cache_hits = r->r.cache_hits;
}

}  // extern "C"
