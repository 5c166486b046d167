"""Univariate programs (gtu_program_*, genfer_b200.UniProgram): a DAG of TaylorExpansion<F64> ops recorded on the host and
run by one launch of k_uni_program.  Every op must give the bits of the per-op gtu_* call of the same name, with the same
variant, order and errors; the symbolic mode (`-s`) evaluates through it in at most three launches."""
import os

import numpy as np
import pytest

gpu = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SYM = os.path.join(HERE, "golden", "sgcl_symbolic")

ORDERS = [1, 2, 31, 32, 33, 34, 35, 64, 257, 1000, 2048]
POW_EXPS = [0, 1, 2, 5, 8]
BINARY = ["add", "sub", "mul", "div", "max"]
UNARY = ["neg", "exp", "log"]
GTP_ERR_INDEX, GTP_ERR_ARG = 1, 5


@pytest.fixture(scope="module")
def G():
    import genfer_b200
    ctx = genfer_b200.Context(0)
    yield genfer_b200, ctx
    ctx.close()


def assert_bits(got, want, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), what
    assert np.array_equal(got[~nan].view(np.int64), want[~nan].view(np.int64)), what


# ---- the same DAG through either path --------------------------------------------------------------------------------
# A node is ("const", x) | ("coeffs", array) | (op, i, j) for op in BINARY | (op, i) for op in UNARY | ("pow", i, e).

def host_max(x, y):
    return x if x > y else y   # F64::max as GpuBackend::scalar_max


def eval_per_op(G, nodes):
    """Replays the nodes through the per-op gtu_* calls; returns the TaylorExpansion of every node."""
    genfer_b200, ctx = G
    E = genfer_b200.TaylorExpansion
    vals = []
    for n in nodes:
        k = n[0]
        if k == "const":
            v = E.constant(n[1], ctx)
        elif k == "coeffs":
            v = E.from_coefficients(n[1], ctx)
        elif k == "pow":
            v = vals[n[1]].pow(n[2])
        elif k == "max":
            v = E.constant(host_max(vals[n[1]].coeff(0), vals[n[2]].coeff(0)), ctx)
        elif k in UNARY:
            v = {"neg": lambda a: -a, "exp": lambda a: a.exp(), "log": lambda a: a.log()}[k](vals[n[1]])
        else:
            a, b = vals[n[1]], vals[n[2]]
            v = {"add": a.__add__, "sub": a.__sub__, "mul": a.__mul__, "div": a.__truediv__}[k](b)
        vals.append(v)
    return vals


def record(G, nodes):
    """Records the nodes into one UniProgram; returns (program, slots)."""
    genfer_b200, ctx = G
    p = genfer_b200.UniProgram(ctx)
    slots = []
    for n in nodes:
        k = n[0]
        if k == "const":
            s = p.constant(n[1])
        elif k == "coeffs":
            s = p.from_coefficients(n[1])
        elif k == "pow":
            s = slots[n[1]].pow(n[2])
        elif k == "max":
            s = slots[n[1]].max(slots[n[2]])
        elif k in UNARY:
            s = {"neg": lambda a: -a, "exp": lambda a: a.exp(), "log": lambda a: a.log()}[k](slots[n[1]])
        else:
            a, b = slots[n[1]], slots[n[2]]
            s = {"add": a.__add__, "sub": a.__sub__, "mul": a.__mul__, "div": a.__truediv__}[k](b)
        slots.append(s)
    return p, slots


def check_same(G, nodes, check_launches=True):
    genfer_b200, ctx = G
    ref = eval_per_op(G, nodes)
    p, slots = record(G, nodes)
    for r, s in zip(ref, slots):
        assert s.is_const() == r.is_const()
        assert s.order() == r.order()
    l0 = ctx.launch_count
    got = p.run(*slots)
    if check_launches:
        assert ctx.launch_count - l0 == 1
    for i, (r, g) in enumerate(zip(ref, got)):
        assert_bits(g, r.coeffs(), f"node {i}: {nodes[i][0]}")


# ---- 1. op matrix ----------------------------------------------------------------------------------------------------

def operand(rng, n, zero_first=False):
    if n is None:
        return ("const", 0.0 if zero_first else float(rng.uniform(0.5, 1.5)))
    xs = rng.uniform(-1.0, 1.0, n) * 0.9 ** np.arange(n)
    xs[0] = 0.0 if zero_first else rng.uniform(0.5, 1.5)
    return ("coeffs", xs)


def binary_cases():
    out = []
    for op in BINARY:
        if op == "max":
            out.append((op, None, None))
            continue
        out.append((op, None, None))
        for n in ORDERS:
            out += [(op, n, None), (op, None, n), (op, n, n)]
        out.append((op, 33, 257))   # operands of different orders: truncated to the shorter
        out.append((op, 2048, 31))
    return out


@gpu
@pytest.mark.parametrize("op,na,nb", binary_cases())
def test_binary_op_matches_per_op_call(G, op, na, nb):
    rng = np.random.default_rng([BINARY.index(op), na or 0, nb or 0])
    check_same(G, [operand(rng, na), operand(rng, nb), (op, 0, 1)])
    if op == "div":   # a divisor with a zero constant term: inf / nan in the same places
        check_same(G, [operand(rng, na), operand(rng, nb, zero_first=True), (op, 0, 1)])


@gpu
@pytest.mark.parametrize("op", UNARY)
@pytest.mark.parametrize("n", [None] + ORDERS)
def test_unary_op_matches_per_op_call(G, op, n):
    rng = np.random.default_rng([UNARY.index(op), n or 0])
    check_same(G, [operand(rng, n), (op, 0)])
    if op == "log":
        check_same(G, [operand(rng, n, zero_first=True), (op, 0)])


@gpu
@pytest.mark.parametrize("e", POW_EXPS)
@pytest.mark.parametrize("n", [None] + ORDERS)
def test_pow_matches_per_op_call(G, n, e):
    rng = np.random.default_rng([e, n or 0])
    check_same(G, [operand(rng, n), ("pow", 0, e)])


@gpu
def test_max_of_constants(G):
    genfer_b200, ctx = G
    cases = [(1.0, 2.0), (2.0, 1.0), (-0.0, 0.0), (0.0, -0.0), (float("nan"), 1.0), (1.0, float("nan"))]
    p = genfer_b200.UniProgram(ctx)
    slots = [p.constant(x).max(p.constant(y)) for x, y in cases]
    for (x, y), g in zip(cases, p.run(*slots)):
        assert_bits(g, [host_max(x, y)])


@gpu
def test_var_input_and_empty_program(G):
    genfer_b200, ctx = G
    E = genfer_b200.TaylorExpansion
    p = genfer_b200.UniProgram(ctx)
    x = p.var(0.5, 40)
    y = (x * x).exp()
    l0 = ctx.launch_count
    gx, gy = p.run(x, y)
    assert ctx.launch_count - l0 == 1
    ex = E.var(0.5, 40, ctx)
    assert_bits(gx, ex.coeffs())
    assert_bits(gy, (ex * ex).exp().coeffs())
    l0 = ctx.launch_count
    assert p.run() == []
    assert ctx.launch_count - l0 == 1


# ---- 2. random DAGs --------------------------------------------------------------------------------------------------

def random_dag(seed, n_ops=300, lo=5, hi=60, top=None):
    """A seeded DAG of `n_ops` mixed ops over polynomial inputs of orders lo..hi (one input of order `top` when given):
    first a level of 40 independent ops, then a chain of 210 dependent steps, then random ops.  Inputs decay
    geometrically and the chain rescales, so most coefficients stay finite."""
    rng = np.random.default_rng(seed)
    nodes = []
    polys, consts = [], []

    def add(n):
        nodes.append(n)
        return len(nodes) - 1

    orders = list(rng.integers(lo, hi + 1, 10))
    if top:
        orders[0] = top
    for n in orders:
        xs = rng.uniform(-1.0, 1.0, n) * 0.7 ** np.arange(n)
        xs[0] = rng.uniform(0.5, 1.5)
        polys.append(add(("coeffs", xs)))
    for _ in range(4):
        consts.append(add(("const", float(rng.uniform(0.5, 2.0)))))
    ops = 0

    def op(n):
        nonlocal ops
        ops += 1
        return add(n)

    leaves = polys + consts
    for i in range(40):   # one wide level
        a, b = rng.choice(leaves, 2)
        kind = ["add", "sub", "mul", "div", "max", "neg", "exp", "log", "pow"][i % 9]
        if kind == "max":
            op(("max", consts[i % 4], consts[(i + 1) % 4]))
        elif kind in ("neg", "exp"):
            op((kind, int(a)))
        elif kind == "log":
            op(("log", polys[i % len(polys)]))
        elif kind == "pow":
            op(("pow", int(a), int(rng.integers(0, 5))))
        elif kind == "div":
            op(("div", int(a), polys[i % len(polys)]))
        else:
            op((kind, int(a), int(b)))
    cur = polys[0]
    half = add(("const", 0.5))
    for i in range(210):   # a chain deeper than 200 levels
        other = int(rng.choice(polys))
        step = i % 7
        if step == 0:
            cur = op(("add", cur, other))
        elif step == 1:
            cur = op(("mul", cur, half))
        elif step == 2:
            cur = op(("sub", cur, other))
        elif step == 3:
            cur = op(("div", cur, other))
        elif step == 4:
            cur = op(("mul", cur, other))
        elif step == 5:
            cur = op(("exp", op(("mul", cur, half))))
        else:
            cur = op(("log", cur))
    while ops < n_ops:   # random ops over everything so far
        a, b = (int(v) for v in rng.integers(0, len(nodes), 2))
        kind = ["add", "sub", "mul", "neg", "div"][int(rng.integers(0, 5))]
        if kind == "neg":
            op(("neg", a))
        elif kind == "div":
            op(("div", a, int(rng.choice(polys))))
        else:
            op((kind, a, b))
    return nodes


def dag_shape(nodes):
    """(levels, maximum level width) of the ops of a node list, levels as the program kernel counts them."""
    level = []
    for n in nodes:
        if n[0] in ("const", "coeffs"):
            level.append(0)
        else:
            args = [n[1]] + ([n[2]] if n[0] in BINARY else [])
            level.append(1 + max(level[a] for a in args))
    ops = [lv for lv in level if lv > 0]
    return max(ops), max(ops.count(lv) for lv in set(ops))


DAG_SEEDS = [(1, None), (2, None), (3, None), (4, 500)]


def test_random_dag_shape_needs_no_gpu():
    for seed, top in DAG_SEEDS:
        levels, width = dag_shape(random_dag(seed, top=top))
        assert levels > 200 and width > 32


@gpu
@pytest.mark.parametrize("seed,top", DAG_SEEDS)
def test_random_dag_matches_per_op_replay(G, seed, top):
    check_same(G, random_dag(seed, top=top))


# ---- 3. errors -------------------------------------------------------------------------------------------------------

@gpu
def test_record_time_errors_launch_nothing(G):
    genfer_b200, ctx = G
    p = genfer_b200.UniProgram(ctx)
    c = p.constant(2.0)
    x = p.var(1.0, 10)
    big = p.var(1.0, 2048)   # 2049 coefficients
    l0 = ctx.launch_count
    with pytest.raises(genfer_b200.TaylorPanic) as e:
        x.max(c)
    assert e.value.status == GTP_ERR_INDEX
    with pytest.raises(genfer_b200.TaylorPanic):
        c.max(x)
    with pytest.raises(genfer_b200.TaylorError) as e:
        p.op(0, x, genfer_b200.UniSlot(p, 10_000))
    assert e.value.status == GTP_ERR_ARG
    with pytest.raises(genfer_b200.TaylorError) as e:
        p.op(5, genfer_b200.UniSlot(p, 10_000))
    assert e.value.status == GTP_ERR_ARG
    with pytest.raises(genfer_b200.TaylorError) as e:
        c / big
    assert e.value.status == GTP_ERR_ARG
    with pytest.raises(genfer_b200.TaylorError) as e:
        big / big
    assert e.value.status == GTP_ERR_ARG
    assert ctx.launch_count == l0
    with pytest.raises(genfer_b200.TaylorError) as e:   # the per-op call agrees
        genfer_b200.TaylorExpansion.var(1.0, 2048, ctx) / genfer_b200.TaylorExpansion.var(1.0, 2048, ctx)
    assert e.value.status == GTP_ERR_ARG
    # nothing was recorded by the failed calls: the program still runs
    l0 = ctx.launch_count
    assert p.run(c)[0][0] == 2.0
    assert ctx.launch_count - l0 == 1


def test_null_arguments_are_rejected_without_a_device():
    """Recording needs no device: a program made without a context rejects null handles and out-pointers."""
    import ctypes as C
    import genfer_b200
    lib = genfer_b200.load()
    p, s = C.c_void_p(), C.c_uint32()
    assert lib.gtu_program_create(None, None) == GTP_ERR_ARG
    assert lib.gtu_program_create(None, C.byref(p)) == 0
    try:
        assert lib.gtu_program_constant(None, None, 1.0, C.byref(s)) == GTP_ERR_ARG
        assert lib.gtu_program_constant(None, p, 1.0, None) == GTP_ERR_ARG
        assert lib.gtu_program_var(None, p, 1.0, 4, None) == GTP_ERR_ARG
        assert lib.gtu_program_from_coefficients(None, None, None, 0, C.byref(s)) == GTP_ERR_ARG
        assert lib.gtu_program_constant(None, p, 1.0, C.byref(s)) == 0
        assert lib.gtu_program_op(None, None, 4, s.value, 0, 0, C.byref(s)) == GTP_ERR_ARG
        assert lib.gtu_program_op(None, p, 4, s.value, 0, 0, None) == GTP_ERR_ARG
        assert lib.gtu_program_slot(None, 0, None, None) == GTP_ERR_ARG
        assert lib.gtu_program_slot(p, 1, None, None) == GTP_ERR_ARG
        out = (C.c_double * 1)()
        assert lib.gtu_program_run(None, p, (C.c_uint32 * 1)(0), 1, out) == GTP_ERR_ARG
    finally:
        lib.gtu_program_free(None, p)


# ---- 4. the symbolic mode end to end ---------------------------------------------------------------------------------

def sym_fixtures():
    return sorted(f for f in os.listdir(SYM) if f.endswith(".sgcl"))


def flags_of(src):
    from genfer_b200.evaluator import parse_flags
    o = parse_flags(src)
    return dict(limit=o["limit"], no_probs=o["no_probs"], no_simplify_gf=o["no_simplify_gf"], unroll=o["unroll"])


@gpu
@pytest.mark.parametrize("name", sym_fixtures())
def test_symbolic_mode_runs_in_three_launches(G, name):
    """The symbolic evaluation is one program run each for the rest, the moments and the probabilities.  GenFun::simplify,
    which runs before it in the default mode (shared with Taylor mode), launches multivariate kernels of its own; without
    it the report is the same and only the three program runs remain."""
    genfer_b200, ctx = G
    src = open(os.path.join(SYM, name)).read()
    expect = open(os.path.join(SYM, name[:-5] + ".expect")).read()
    kw = flags_of(src)
    assert genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **kw).report == expect
    kw["no_simplify_gf"] = True
    l0 = ctx.launch_count
    g = genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **kw)
    assert ctx.launch_count - l0 == 3
    assert g.report == expect
    l0 = ctx.launch_count
    genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **dict(kw, no_probs=True))
    assert ctx.launch_count - l0 == 2
