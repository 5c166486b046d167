// C ABI for the univariate TaylorExpansion<F64> (src/univariate_taylor.rs): enum dispatch on the
// host (Constant vs Polynomial), arithmetic on the device.
#include "kernels.cuh"

using namespace gtp;
using SerP = std::unique_ptr<gtu_series>;

namespace {

SerP new_series(Ctx& c, bool is_const, u64 n) {
  SerP s(new gtu_series());
  s->is_const = is_const;
  s->n = is_const ? 1 : n;
  s->buf = c.alloc(std::max<u64>(s->n, 1));
  return s;
}
SerP share(const gtu_series& a) { return SerP(new gtu_series(a)); }

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

// One op through the per-op kernels (uni_plan holds the Constant/Polynomial rules)
SerP uni_op(Ctx& c, int op, const gtu_series& a, const gtu_series* b) {
  const UniPlan p = uni_plan(op, a.is_const, a.n, b && b->is_const, b ? b->n : 0);
  SerP r = new_series(c, p.is_const, p.n);
  uni_run(c, p, a.ptr(), b ? b->ptr() : nullptr, r->buf->d);
  return r;
}

SerP uni_const(Ctx& c, double x) {
  SerP r = new_series(c, true, 1);
  launch_fill(c, r->buf->d, 1, x);
  return r;
}

}  // namespace

// A recorded univariate program.  Slot values live in one device arena laid out as [inputs | computed | gathered outputs]:
// an input's offset is fixed when it is recorded (its coefficients are copied into `inputs`), a computed slot's when its op
// is recorded (relative to the end of the inputs).  Ops are kept with their kernel operands already ordered (UniPlan::swap).
struct gtu_program {
  struct Slot {
    bool is_const;
    u64 n;            // 1 for a Constant
    bool input;
    u64 off;          // doubles, in the inputs or the computed region
    unsigned level;   // 0 for inputs, else one plus the deepest operand
  };
  struct Op {
    UniPlan plan;
    uint32_t x, y, r;   // slots of the kernel's operands (y: UNI_NONE for unary ops) and of the result
  };
  std::vector<Slot> slots;
  std::vector<double> inputs;
  u64 computed = 0;
  std::vector<Op> ops;

  const Slot& at(uint32_t s) const {
    GTP_CHECK(s < slots.size(), GTP_ERR_ARG, "univariate program: slot out of range");
    return slots[s];
  }
  uint32_t add_input(bool is_const, const double* xs, u64 n) {
    GTP_CHECK(slots.size() < UNI_NONE, GTP_ERR_ARG, "univariate program: too many slots");
    slots.push_back({is_const, n, true, (u64)inputs.size(), 0});
    inputs.insert(inputs.end(), xs, xs + n);
    return (uint32_t)slots.size() - 1;
  }
  uint32_t add_op(int op, uint32_t a, uint32_t b) {
    const bool binary = op == GTU_ADD || op == GTU_SUB || op == GTU_MUL || op == GTU_DIV || op == GTU_MAX;
    const Slot sa = at(a);
    const Slot sb = binary ? at(b) : Slot{false, 0, false, 0, 0};
    GTP_CHECK(slots.size() < UNI_NONE, GTP_ERR_ARG, "univariate program: too many slots");
    const UniPlan p = uni_plan(op, sa.is_const, sa.n, sb.is_const, sb.n);
    const uint32_t y = binary ? b : UNI_NONE;
    slots.push_back({p.is_const, p.n, false, computed, 1 + std::max(sa.level, sb.level)});
    computed += p.n;
    ops.push_back({p, p.swap ? y : a, p.swap ? a : y, (uint32_t)slots.size() - 1});
    return ops.back().r;
  }
  uint32_t add_pow(uint32_t a, uint32_t e) {   // gtu_pow's products, including the last (unused) squaring
    at(a);
    const double one = 1.0;
    uint32_t res = add_input(true, &one, 1), base = a;
    while (e > 0) {
      if (e & 1) res = add_op(GTU_MUL, res, base);
      base = add_op(GTU_MUL, base, base);
      e >>= 1;
    }
    return res;
  }
  u64 arena_off(uint32_t s) const { return slots[s].input ? slots[s].off : inputs.size() + slots[s].off; }

  void run(Ctx& c, const uint32_t* outputs, int n_outputs, double* out) {
    GTP_CHECK(n_outputs >= 0 && (outputs || n_outputs == 0), GTP_ERR_ARG, "univariate program: bad output list");
    const u64 n_in = inputs.size(), gather = n_in + computed;
    u64 n_out = 0;
    std::vector<unsigned> outs;
    for (int o = 0; o < n_outputs; o++) {
      const Slot& s = at(outputs[o]);
      outs.insert(outs.end(), {(unsigned)arena_off(outputs[o]), (unsigned)s.n, (unsigned)(gather + n_out)});
      n_out += s.n;
    }
    GTP_CHECK(out || n_out == 0, GTP_ERR_ARG, "null output");
    GTP_CHECK(gather + n_out < UNI_NONE, GTP_ERR_ARG, "univariate program: arena larger than 2^32 doubles");

    // levels, and each level's ops dealt to warps longest first (LPT: the next op goes to the least loaded warp)
    unsigned nlevels = 0;
    for (const Op& op : ops) nlevels = std::max(nlevels, slots[op.r].level);
    std::vector<std::vector<uint32_t>> by_level(nlevels);
    for (uint32_t i = 0; i < ops.size(); i++) by_level[slots[ops[i].r].level - 1].push_back(i);
    size_t width = 1;
    for (const auto& l : by_level) width = std::max(width, l.size());
    const unsigned nw = (unsigned)std::min<size_t>(width, 32);
    auto cost = [&](const Op& op) -> u64 {
      const u64 n = op.plan.n;
      return op.plan.kind == UK_EW ? n : (op.plan.kind == UK_SCALAR_EXP || op.plan.kind == UK_SCALAR_LOG) ? 1 : n * n;
    };
    std::vector<UniIns> ins;
    ins.reserve(ops.size());
    std::vector<unsigned> lvl{0};
    lvl.reserve((u64)nlevels * nw + 1);
    for (auto& l : by_level) {
      std::stable_sort(l.begin(), l.end(), [&](uint32_t i, uint32_t j) { return cost(ops[i]) > cost(ops[j]); });
      std::vector<u64> load(nw, 0);
      std::vector<std::vector<uint32_t>> dealt(nw);
      for (uint32_t i : l) {
        const unsigned w = (unsigned)(std::min_element(load.begin(), load.end()) - load.begin());
        load[w] += cost(ops[i]) + 1;
        dealt[w].push_back(i);
      }
      for (const auto& d : dealt) {
        for (uint32_t i : d) {
          const Op& op = ops[i];
          UniIns u{};
          u.a = (unsigned)arena_off(op.x);
          u.b = op.y == UNI_NONE ? UNI_NONE : (unsigned)arena_off(op.y);
          u.r = (unsigned)arena_off(op.r);
          u.n = (unsigned)op.plan.n;
          u.kind = (unsigned char)op.plan.kind;
          u.ew = (unsigned char)op.plan.ew;
          u.a_b = op.plan.a_b;
          u.b_b = op.plan.b_b;
          ins.push_back(u);
        }
        lvl.push_back((unsigned)ins.size());
      }
    }

    // one upload: [ins | lvl | outs | pad] then the inputs, which start the arena
    const u64 tab_bytes = ins.size() * sizeof(UniIns) + (lvl.size() + outs.size()) * sizeof(unsigned);
    const u64 tab = (tab_bytes + sizeof(double) - 1) / sizeof(double);
    double* host = c.host_staging(std::max(tab + n_in, n_out));
    char* h = reinterpret_cast<char*>(host);
    std::memcpy(h, ins.data(), ins.size() * sizeof(UniIns));
    std::memcpy(h + ins.size() * sizeof(UniIns), lvl.data(), lvl.size() * sizeof(unsigned));
    std::memcpy(h + ins.size() * sizeof(UniIns) + lvl.size() * sizeof(unsigned), outs.data(), outs.size() * sizeof(unsigned));
    if (n_in) std::memcpy(host + tab, inputs.data(), n_in * sizeof(double));
    BufP dev = c.alloc(tab + gather + n_out);
    char* d = reinterpret_cast<char*>(dev->d);
    GTP_CUDA(cudaMemcpyAsync(d, host, (tab + n_in) * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    const UniIns* d_ins = reinterpret_cast<const UniIns*>(d);
    const unsigned* d_lvl = reinterpret_cast<const unsigned*>(d + ins.size() * sizeof(UniIns));
    uni_program_launch(c, d_ins, d_lvl, (int)nlevels, (int)nw, d_lvl + lvl.size(), n_outputs, dev->d + tab);
    if (n_out) GTP_CUDA(cudaMemcpyAsync(host, dev->d + tab + gather, n_out * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    if (n_out) std::memcpy(out, host, n_out * sizeof(double));
  }
};

extern "C" {

int gtu_constant(gtp_ctx* c, double x, gtu_series** out) { return wrap(c, [&] { *out = uni_const(*c, x).release(); }); }
int gtu_from_coefficients(gtp_ctx* c, const double* xs, uint64_t n, gtu_series** out) {
  return wrap(c, [&] {
    GTP_CHECK(xs || n == 0, GTP_ERR_ARG, "null coefficients");
    SerP r = new_series(*c, false, n);
    if (n) GTP_CUDA(cudaMemcpyAsync(r->buf->d, xs, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    *out = r.release();
  });
}
int gtu_var(gtp_ctx* c, double x, uint64_t order, gtu_series** out) {  // :16-23
  return wrap(c, [&] {
    std::vector<double> v(order + 1, 0.0);
    if (v.size() > 1) v[1] = 1.0;
    v[0] = x;
    SerP r = new_series(*c, false, order + 1);
    GTP_CUDA(cudaMemcpyAsync(r->buf->d, v.data(), v.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    c->sync();  // `v` is pageable and dies at scope exit
    *out = r.release();
  });
}
void gtu_free(gtp_ctx* c, gtu_series* s) {
  if (c) cudaSetDevice(c->device);
  delete s;
}
int gtu_is_constant(const gtu_series* s) { return s->is_const ? 1 : 0; }
uint64_t gtu_order(const gtu_series* s) { return s->is_const ? GTP_UNBOUNDED : s->n; }
int gtu_to_host(gtp_ctx* c, const gtu_series* s, double* out) {
  return wrap(c, [&] {
    if (s->n) GTP_CUDA(cudaMemcpyAsync(out, s->ptr(), s->n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
  });
}
int gtu_coeff(gtp_ctx* c, const gtu_series* s, uint64_t order, double* out) {  // :25-36
  return wrap(c, [&] {
    if (s->is_const && order != 0) { *out = 0.0; return; }
    GTP_CHECK(s->is_const || order < s->n, GTP_ERR_INDEX, "coeff: index out of bounds");
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], s->ptr() + (s->is_const ? 0 : order), sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
    *out = c->rb_host->vals[0];
  });
}
int gtu_derivative(gtp_ctx* c, const gtu_series* s, uint64_t order, double* out) {  // :45-60
  return wrap(c, [&] {
    if (s->is_const) {
      if (order != 0) { *out = 0.0; return; }
      GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], s->ptr(), sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    } else {
      GTP_CHECK(order < s->n, GTP_ERR_INDEX, "derivative: index out of bounds");
      uni_factorial_times(*c, s->ptr(), order, &c->rb_dev->vals[0]);
      GTP_CUDA(cudaMemcpyAsync(&c->rb_host->vals[0], &c->rb_dev->vals[0], sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    c->sync();
    *out = c->rb_host->vals[0];
  });
}
int gtu_add(gtp_ctx* c, const gtu_series* a, const gtu_series* b, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_ADD, *a, b).release(); }); }
int gtu_sub(gtp_ctx* c, const gtu_series* a, const gtu_series* b, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_SUB, *a, b).release(); }); }
int gtu_mul(gtp_ctx* c, const gtu_series* a, const gtu_series* b, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_MUL, *a, b).release(); }); }
int gtu_div(gtp_ctx* c, const gtu_series* a, const gtu_series* b, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_DIV, *a, b).release(); }); }
int gtu_neg(gtp_ctx* c, const gtu_series* a, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_NEG, *a, nullptr).release(); }); }  // :308-319
int gtu_exp(gtp_ctx* c, const gtu_series* a, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_EXP, *a, nullptr).release(); }); }  // :151-168
int gtu_log(gtp_ctx* c, const gtu_series* a, gtu_series** out) { return wrap(c, [&] { *out = uni_op(*c, GTU_LOG, *a, nullptr).release(); }); }  // :170-189
int gtu_pow(gtp_ctx* c, const gtu_series* a, uint32_t e, gtu_series** out) {  // :192-203
  return wrap(c, [&] {
    SerP res = uni_const(*c, 1.0);
    SerP base = share(*a);
    while (e > 0) {
      if (e & 1) res = uni_op(*c, GTU_MUL, *res, base.get());
      base = uni_op(*c, GTU_MUL, *base, base.get());
      e >>= 1;
    }
    *out = res.release();
  });
}
int gtu_subst(gtp_ctx* c, const gtu_series* a, const gtu_series* s, gtu_series** out) {  // :93-115
  return wrap(c, [&] {
    if (a->is_const) { *out = share(*a).release(); return; }
    if (!s->is_const) GTP_CHECK(s->n == a->n, GTP_ERR_INDEX, "Substitution must have the same order");
    SerP res = uni_const(*c, 0.0);
    for (u64 i = a->n; i-- > 0;) {
      SerP p = uni_op(*c, GTU_MUL, *res, s);
      gtu_series ci;  // Constant(c_i) viewed in place
      ci.is_const = true;
      ci.n = 1;
      auto b = std::make_shared<Buf>();
      b->d = const_cast<double*>(a->ptr() + i);
      b->n = 1;
      b->owned = false;
      ci.buf = b;
      res = uni_op(*c, GTU_ADD, *p, &ci);
    }
    *out = res.release();
  });
}
int gtu_taylor_expansion_of_coeff(gtp_ctx* c, const gtu_series* a, uint64_t n, gtu_series** out) {  // :69-89
  return wrap(c, [&] {
    if (a->is_const) {
      if (n == 0) {  // sic: the reference returns Constant(c.exp()) here (:73)
        SerP r = new_series(*c, true, 1);
        launch_scalar_fn(*c, 0, a->ptr(), r->buf->d);
        *out = r.release();
      } else {
        *out = uni_const(*c, 0.0).release();
      }
      return;
    }
    GTP_CHECK(n <= a->n, GTP_ERR_INDEX, "taylor_expansion_of_coeff: slice start out of range");
    SerP r = new_series(*c, false, a->n - n);
    uni_teoc(*c, a->ptr(), r->buf->d, n, a->n - n);
    *out = r.release();
  });
}
int gtu_eq(gtp_ctx* c, const gtu_series* a, const gtu_series* b, int* out) {
  return wrap(c, [&] {
    *out = 0;
    if (a->is_const != b->is_const || a->n != b->n) return;
    if (a->n == 0) { *out = 1; return; }
    launch_eq(*c, a->ptr(), b->ptr(), a->n, c->rb_dev);
    GTP_CUDA(cudaMemcpyAsync(&c->rb_host->flag, &c->rb_dev->flag, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    c->sync();
    *out = c->rb_host->flag ? 1 : 0;
  });
}

int gtu_program_create(gtp_ctx* c, gtu_program** out) {
  return wrap(c, [&] {
    GTP_CHECK(out, GTP_ERR_ARG, "null argument");
    *out = new gtu_program();
  });
}
void gtu_program_free(gtp_ctx*, gtu_program* p) { delete p; }
int gtu_program_constant(gtp_ctx* c, gtu_program* p, double x, uint32_t* slot) {
  return wrap(c, [&] {
    GTP_CHECK(p && slot, GTP_ERR_ARG, "null argument");
    *slot = p->add_input(true, &x, 1);
  });
}
int gtu_program_var(gtp_ctx* c, gtu_program* p, double x, uint64_t order, uint32_t* slot) {  // :16-23
  return wrap(c, [&] {
    GTP_CHECK(p && slot, GTP_ERR_ARG, "null argument");
    std::vector<double> v(order + 1, 0.0);
    if (v.size() > 1) v[1] = 1.0;
    v[0] = x;
    *slot = p->add_input(false, v.data(), v.size());
  });
}
int gtu_program_from_coefficients(gtp_ctx* c, gtu_program* p, const double* xs, uint64_t n, uint32_t* slot) {
  return wrap(c, [&] {
    GTP_CHECK(p && slot, GTP_ERR_ARG, "null argument");
    GTP_CHECK(xs || n == 0, GTP_ERR_ARG, "null coefficients");
    *slot = p->add_input(false, xs, n);
  });
}
int gtu_program_op(gtp_ctx* c, gtu_program* p, int op, uint32_t a, uint32_t b, uint32_t exp, uint32_t* slot) {
  return wrap(c, [&] {
    GTP_CHECK(p && slot, GTP_ERR_ARG, "null argument");
    *slot = op == GTU_POW ? p->add_pow(a, exp) : p->add_op(op, a, b);
  });
}
int gtu_program_slot(const gtu_program* p, uint32_t slot, int* is_constant, uint64_t* n) {
  return wrap(nullptr, [&] {
    GTP_CHECK(p, GTP_ERR_ARG, "null argument");
    const gtu_program::Slot& s = p->at(slot);
    if (is_constant) *is_constant = s.is_const ? 1 : 0;
    if (n) *n = s.is_const ? GTP_UNBOUNDED : s.n;
  });
}
int gtu_program_run(gtp_ctx* c, gtu_program* p, const uint32_t* outputs, int n_outputs, double* out) {
  return wrap(c, [&] {
    GTP_CHECK(c && p, GTP_ERR_ARG, "null argument");
    p->run(*c, outputs, n_outputs, out);
  });
}

}  // extern "C"
