"""Truncated products, the operators built on them and the interval type on tensors with 9 to 24 non-unit axes.

From 2^20 MACs such products run on the trailing-box DFMA kernel (k_mul_box, plan kind 8: another summation order, 1e-12
like the other DFMA kernels, exact on small integers); below that, and with set_fast_mul(0), on the reference-order kernel
(k_mul_ordered<NE>, NE up to GTP_MAX_NDIM; k_mul_ordered_cls<9|10> for results of at most 1024 coefficients), in the
reference's summation order: bit-identical to the oracle.  Products are checked on small-integer operands (every partial sum
exact, whatever the order) and on random doubles, by the full result or by a row sample where the oracle would take minutes.  The operators are held to the tolerances the rest of the suite applies to
them at fewer axes; the interval product is bit-identical to the oracle's Interval<F64> instantiation and the interval
recurrences enclose the f64 result.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_bits, assert_close, assert_same, small_ints

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
MODES = [1, 0]   # gtp_ctx_set_fast_mul: fastest applicable route (default), reference-order kernel only


@pytest.fixture(scope="module")
def G():
    import genfer_b200
    ctx = genfer_b200.Context(0)
    genfer_b200.set_default_context(ctx)
    yield genfer_b200
    genfer_b200.set_default_context(None)
    ctx.close()


def O():
    from oracle import oracle
    return oracle


def device_product(ctx, mode, x, y, rshape, rows=None, row_list=None):
    """gtp_mul_rows_raw (rows = (begin, step, count), default all) or gtp_mul_rowlist_raw (row_list) on device buffers."""
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    yd = torch.from_numpy(np.ascontiguousarray(y)).cuda()
    count = len(row_list) if row_list is not None else (rows[2] if rows else rshape[0])
    out = torch.full((count,) + tuple(rshape[1:]), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.set_fast_mul(mode)
    try:
        if row_list is not None:
            ctx.mul_rowlist_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, row_list, out.data_ptr())
        else:
            begin, step, n = rows if rows else (0, 1, rshape[0])
            ctx.mul_rows_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, begin, step, n, out.data_ptr())
        ctx.synchronize()
    finally:
        ctx.set_fast_mul(1)
    return out.cpu().numpy()


def nonunit(shape):
    return sum(e != 1 for e in shape)


# (xs, ys, rs): ragged extents 2..4, unit axes in between, operands of different extents, result degrees that truncate some
# axes.  At 16 and 24 axes one operand has extent 1 on most axes: the result axis stays non-unit at one MAC per output.
PRODUCTS = [
    ((2,) * 9, (2,) * 9, (3,) * 9),
    ((3, 2, 4, 1, 2, 3, 2, 2, 3, 2), (2, 3, 2, 1, 3, 2, 2, 3, 2, 2), (4, 4, 3, 1, 4, 4, 3, 3, 4, 3)),
    ((3,) * 10, (3,) * 10, (3,) * 10),
    ((2, 3, 2, 2, 1, 2, 2, 3, 2, 2, 2, 2, 2), (3, 2, 2, 2, 1, 2, 2, 2, 2, 3, 2, 2, 2), (4, 3, 3, 2, 1, 3, 3, 3, 3, 4, 2, 3, 3)),
    ((2,) * 16, (1,) * 12 + (3, 2, 3, 2), (2,) * 12 + (4, 3, 3, 3)),
    ((1,) * 13 + (2, 4, 3), (3, 2) * 8, (3, 2) * 6 + (3, 2, 4, 4)),
    ((2,) * 24, (1,) * 20 + (2, 3, 2, 2), (2,) * 24),
]
assert sorted({nonunit(rs) for _, _, rs in PRODUCTS}) == [9, 10, 12, 16, 24]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("xs,ys,rs", PRODUCTS, ids=lambda s: "x".join(map(str, s)))
def test_product_small_ints_bit_exact(G, mode, xs, ys, rs):
    x, y = small_ints(xs, 91), small_ints(ys, 92)
    assert_bits(device_product(G.default_context(), mode, x, y, rs), O().mul_raw(x, y, rs))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("xs,ys,rs", PRODUCTS, ids=lambda s: "x".join(map(str, s)))
def test_product_random_doubles(G, mode, xs, ys, rs):
    rng = np.random.default_rng(nonunit(rs) * 7 + mode)
    x, y = rng.uniform(-1.0, 1.0, xs), rng.uniform(-1.0, 1.0, ys)
    got, ref = device_product(G.default_context(), mode, x, y, rs), O().mul_raw(x, y, rs)
    if mode == 0:
        assert_bits(got, ref)
    scale = np.abs(ref).max()
    assert np.all(np.abs(got - ref) <= 1e-12 * (np.abs(ref) + scale))


@pytest.mark.parametrize("mode", MODES)
def test_product_row_ranges_and_lists_10_axes(G, mode):
    """Row subsets as group contexts issue them: a range with a step (the cyclic partition) and a folded-cyclic row list
    (genfer_b200.partition.rows_for_rank) on a 10-axis product."""
    from genfer_b200.partition import rows_for_rank
    xs = ys = rs = (8,) + (3,) * 9
    x, y = small_ints(xs, 93), small_ints(ys, 94)
    ref = O().mul_raw(x, y, rs)
    ctx = G.default_context()
    assert_bits(device_product(ctx, mode, x, y, rs, rows=(1, 3, 3)), ref[1:8:3])
    for rank in range(3):
        rows = rows_for_rank(8, 3, rank)
        assert_bits(device_product(ctx, mode, x, y, rs, row_list=rows), ref[rows])
    assert_bits(device_product(ctx, mode, x, y, rs, row_list=[6, 2, 4, 5]), ref[[6, 2, 4, 5]])


@pytest.mark.parametrize("mode", MODES)
def test_dense_product_row_sample(G, mode):
    """[8, 3^9] squared (157 K coefficients, 3.6 * 10^8 MACs) and [4]^10 squared (1.05 M coefficients, 10^10 MACs):
    leading-axis rows against the oracle."""
    rng = np.random.default_rng(95)
    for shape, rows in (((8,) + (3,) * 9, [0, 1, 7]), ((4,) * 10, [0])):
        x, y = rng.uniform(0.0, 1.0, shape), rng.uniform(0.0, 1.0, shape)
        ref, _ = O().mul_rows(x, y, shape, rows)
        got = device_product(G.default_context(), mode, x, y, shape)[rows]
        if mode == 0:
            assert_bits(got, ref[rows])
        assert np.all(np.abs(got - ref[rows]) <= 1e-12 * np.abs(ref[rows]))


def test_small_result_classified_by_the_producer(G):
    """Results of at most 1024 coefficients run on the single-CTA kernel that also classifies its output: a linear and an
    all-zero result at 9 and 10 axes, through TaylorPoly's product (is_zero / extract_linear read that classification)."""
    for n in (9, 10):
        shape = (2,) * n
        z, e0 = np.zeros(shape), np.zeros(shape)
        z[(1, 1) + (0,) * (n - 2)] = 1.0          # a two-variable monomial: neither operand is linear
        e0[(1,) + (0,) * (n - 1)] = 1.0
        one = np.zeros(shape)
        one.flat[0] = 1.0
        # (1 + z)(1 - z + 2 e0) = 1 + 2 e0 and z (z + e0) = 0 once z^2 and z e0 are truncated
        for a, b, linear in ((one + z, one - z + 2.0 * e0, (1.0, 2.0, 0)), (z, z + e0, (0.0, 0.0, 0))):
            for mode in MODES:
                G.default_context().set_fast_mul(mode)
                try:
                    g = G.TaylorPoly.new(a, shape) * G.TaylorPoly.new(b, shape)
                finally:
                    G.default_context().set_fast_mul(1)
                o = O().TaylorPoly.new(a, shape) * O().TaylorPoly.new(b, shape)
                assert_same(g, o)
                assert g.is_zero() == o.is_zero()
                assert g.extract_linear() == o.extract_linear() == linear


# ---------------------------------------------------------------------------------------------------------------------
# the reported kind is the kernel that runs
# ---------------------------------------------------------------------------------------------------------------------
CHILD = r"""
import os, sys, torch
import genfer_b200
for i, (xs, ys, rs) in enumerate(eval(sys.argv[1])):
    os.write(2, b"@@product %d\n" % i)
    ctx = genfer_b200.Context(0)
    kind = ctx.mul_kernel_kind(xs, ys, rs)
    x = torch.ones(xs, dtype=torch.float64, device="cuda")
    y = torch.ones(ys, dtype=torch.float64, device="cuda")
    z = torch.empty(rs, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.mul_rows_raw(xs, x.data_ptr(), ys, y.data_ptr(), rs, 0, 1, rs[0], z.data_ptr())
    ctx.synchronize()
    os.write(2, b"@@kind %d\n" % kind)
    ctx.close()
"""
KIND_SHAPES = PRODUCTS + [((4,) * 10,) * 3, ((3,) * 12,) * 3]


def test_reported_kind_is_the_kernel_that_runs():
    env = dict(os.environ, GTP_LAUNCH_HIST="1")
    env.pop("GTP_FAST_MUL", None)
    r = subprocess.run([sys.executable, "-c", CHILD, repr(KIND_SHAPES)], cwd=REPO, env=env, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    parts = r.stderr.split("@@product ")[1:]
    assert len(parts) == len(KIND_SHAPES)
    for part, (xs, ys, rs) in zip(parts, KIND_SHAPES):
        kind = int(re.search(r"^@@kind (\d+)$", part, re.M).group(1))
        names = set(re.findall(r"^\[gtp launches\]\s+\d+\s+(.+)$", part, re.M))
        ne = nonunit(rs)
        big = O().mul_macs(xs, ys, rs) >= 2 ** 20
        assert kind == (8 if big else 0), (rs, kind)
        if big:
            assert "k_mul_box" in names and not any("k_mul_ordered" in n for n in names), (rs, names)
        else:
            assert names & {f"k_mul_ordered<{ne}>", f"k_mul_ordered_cls<{ne}>"} and "k_mul_box" not in names, (rs, names)
        assert not any("k_mul_slide" in n or "k_mul_blk" in n for n in names), (rs, names)


CLS_CHILD = r"""
import sys
import numpy as np
import genfer_b200
ctx = genfer_b200.Context(0)
for n in (9, 10):
    a = np.zeros((2,) * n); a.flat[0] = 1.0; a.flat[-1] = 2.0; a[(1, 1) + (0,) * (n - 2)] = 3.0
    p = genfer_b200.TaylorPoly.new(a, (2,) * n, ctx)
    q = p * p
    q.is_zero(); q.extract_linear()
ctx.close()
"""


def test_small_results_run_on_the_classifying_kernel():
    """Products of at most 1024 coefficients on 9 and 10 axes launch k_mul_ordered_cls<9> / <10>."""
    env = dict(os.environ, GTP_LAUNCH_HIST="1")
    env.pop("GTP_FAST_MUL", None)
    r = subprocess.run([sys.executable, "-c", CLS_CHILD], cwd=REPO, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    names = set(re.findall(r"^\[gtp launches\]\s+\d+\s+(.+)$", r.stderr, re.M))
    assert {"k_mul_ordered_cls<9>", "k_mul_ordered_cls<10>"} <= names, names


# ---------------------------------------------------------------------------------------------------------------------
# operators
# ---------------------------------------------------------------------------------------------------------------------
OPERANDS = [((2,) * 9, (3,) * 9), ((2, 3, 2, 1, 2, 2, 2, 2, 2, 2), (3, 3, 2, 1, 3, 2, 2, 2, 2, 3)), ((2,) * 10, (2,) * 10)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape,deg", OPERANDS, ids=lambda s: "x".join(map(str, s)))
def test_exp_log_pow_div(G, mode, shape, deg):
    rng = np.random.default_rng(sum(shape) + mode)
    a = rng.uniform(0.5, 1.5, shape)
    b = rng.uniform(-0.3, 0.3, shape)
    b.flat[0] = 2.0
    G.default_context().set_fast_mul(mode)
    try:
        ga, gb = G.TaylorPoly.new(a, deg), G.TaylorPoly.new(b, deg)
        got = {"exp": ga.exp(), "log": ga.log(), "pow5": ga.pow(5), "div": ga / gb}
    finally:
        G.default_context().set_fast_mul(1)
    oa, ob = O().TaylorPoly.new(a, deg), O().TaylorPoly.new(b, deg)
    ref = {"exp": oa.exp(), "log": oa.log(), "pow5": oa.pow(5), "div": oa / ob}
    for name in ("exp", "log", "pow5", "div"):
        assert_close(got[name], ref[name], rtol=1e-12)
    if mode == 0:   # products only, in the reference's order; the exp seed from the host's libm (<= 8192 coefficients)
        assert_same(got["pow5"], ref["pow5"])
        assert_same(got["exp"], ref["exp"])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("shape,deg", OPERANDS, ids=lambda s: "x".join(map(str, s)))
def test_subst_var(G, mode, shape, deg):
    """Horner steps of products (the fused Horner loop stops at 8 axes): bit-exact in exact mode, as at fewer axes."""
    rng = np.random.default_rng(3 * sum(shape) + mode)
    a = rng.uniform(0.1, 1.0, shape)
    dense = rng.uniform(0.1, 1.0, shape)
    small_shape = [1] * len(shape)
    small_shape[1], small_shape[-1] = 2, 2
    small = rng.uniform(0.1, 1.0, small_shape)
    G.default_context().set_fast_mul(mode)
    try:
        g = G.TaylorPoly.new(a, deg)
        got = [g.subst_var(v, G.TaylorPoly.new(s, deg)) for v in (0, len(shape) - 1) for s in (small, dense)]
    finally:
        G.default_context().set_fast_mul(1)
    o = O().TaylorPoly.new(a, deg)
    ref = [o.subst_var(v, O().TaylorPoly.new(s, deg)) for v in (0, len(shape) - 1) for s in (small, dense)]
    for r_g, r_o in zip(got, ref):
        if mode == 0:
            assert_same(r_g, r_o)
        else:   # steps from 2^20 MACs on the DFMA kernel
            assert_close(r_g, r_o, rtol=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# interval type
# ---------------------------------------------------------------------------------------------------------------------
def rand_iv(rng, shape, width=1e-9):
    mid = rng.uniform(-1.0, 1.0, size=shape)
    w = rng.uniform(0.0, width, size=shape)
    return np.stack([mid - w, mid + w], axis=-1)


@pytest.mark.parametrize("xs,ys,deg", [((2,) * 13, (2, 1) * 6 + (3,), (3,) * 13),
                                       ((2,) * 16, (1,) * 13 + (2, 3, 2), (2,) * 13 + (3, 3, 3)),
                                       ((1,) * 10 + (2,) * 4, (3, 2) * 7, (3, 2) * 5 + (3,) * 4)])
def test_interval_product_bit_exact(G, xs, ys, deg):
    from genfer_b200.interval import IntervalPoly
    rng = np.random.default_rng(len(xs) + sum(ys))
    x, y = rand_iv(rng, xs), rand_iv(rng, ys)
    ctx = G.default_context()
    g = IntervalPoly.new(x, deg, ctx) * IntervalPoly.new(y, deg, ctx)
    o = O().TaylorPoly.new(x, deg, "iv") * O().TaylorPoly.new(y, deg, "iv")
    assert nonunit(g.array_shape()) == len(xs)
    assert g.array_shape() == o.array_shape()
    assert np.array_equal(g.array(), o.array(), equal_nan=True)


def test_interval_exp_div_13_axes(G):
    """Overlap with the oracle's enclosure, at most 8x its width, and enclosure of the device's f64 result
    (tests/test_gpu_interval.py's rules)."""
    from genfer_b200.interval import IntervalPoly
    shape = (2,) * 13
    rng = np.random.default_rng(13)
    a = rng.uniform(-0.5, 0.5, size=shape)
    a.flat[0] = 1.5
    b = rng.uniform(-0.3, 0.3, size=shape)
    b.flat[0] = 2.0
    w = 1e-12
    ai, bi = np.stack([a - w, a + w], -1), np.stack([b - w, b + w], -1)
    ctx = G.default_context()
    ga, gb = IntervalPoly.new(ai, shape, ctx), IntervalPoly.new(bi, shape, ctx)
    oa, ob = O().TaylorPoly.new(ai, shape, "iv"), O().TaylorPoly.new(bi, shape, "iv")
    fa, fb = G.TaylorPoly.new(a, shape), G.TaylorPoly.new(b, shape)
    for g, o, point in ((ga.exp(), oa.exp(), fa.exp().array()), (ga / gb, oa / ob, (fa / fb).array())):
        ga_, oa_ = g.array(), o.array()
        assert ga_.shape == oa_.shape
        assert np.all(ga_[..., 0] <= ga_[..., 1])
        assert np.all(np.maximum(ga_[..., 0], oa_[..., 0]) <= np.minimum(ga_[..., 1], oa_[..., 1])), "enclosures do not overlap"
        wg, wo = ga_[..., 1] - ga_[..., 0], oa_[..., 1] - oa_[..., 0]
        tiny = 64 * np.finfo(float).eps * np.maximum(np.abs(oa_).max(axis=-1), 1e-300)
        assert np.all(wg <= 8.0 * wo + tiny), float((wg / (wo + tiny)).max())
        assert np.all((ga_[..., 0] <= point) & (point <= ga_[..., 1])), "f64 result outside the enclosure"


# ---------------------------------------------------------------------------------------------------------------------
# end to end: a program with nine live correlated variables
# ---------------------------------------------------------------------------------------------------------------------
PROGRAM = os.path.join(HERE, "thinning_tree_9vars.sgcl")
RUN_CHILD = r"""
import sys
import genfer_b200
src = open(sys.argv[1]).read()
ctx = genfer_b200.Context(0)
genfer_b200.run_sgcl(src, no_probs=True, ctx=ctx)
ctx.close()
"""


def test_program_issues_products_on_nine_axes():
    """The launch census of the program's evaluation shows a product kernel at nine or more non-unit axes."""
    env = dict(os.environ, GTP_LAUNCH_HIST="1")
    env.pop("GTP_FAST_MUL", None)
    r = subprocess.run([sys.executable, "-c", RUN_CHILD, PROGRAM], cwd=REPO, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    names = re.findall(r"^\[gtp launches\]\s+\d+\s+(k_mul_box|k_mul_ordered(?:_cls)?<\d+>)$", r.stderr, re.M)
    wide = [n for n in names if n == "k_mul_box" or int(n.split("<")[1][:-1]) >= 9]   # k_mul_box: > 8 axes only
    assert wide, names


def test_program_matches_oracle_and_bounds_enclose(G):
    import genfer_b200
    from genfer_b200.interval import run_sgcl_bounds
    from helpers import check_inside_enclosure
    src = open(PROGRAM).read()
    opts = genfer_b200.parse_flags(src)
    ctx = G.default_context()
    g = genfer_b200.run_sgcl(src, limit=opts["limit"], no_probs=opts["no_probs"], ctx=ctx)
    o = O().run_sgcl(src, limit=opts["limit"], no_probs=opts["no_probs"])
    if g.report != o.report:
        assert abs(g.total - o.total) <= 1e-12 * abs(o.total), (g.total, o.total)
        for k, (a, b) in enumerate(zip(g.moments[:5], o.moments[:5])):
            assert abs(a - b) <= 1e-12 * max(abs(b), 1.0), (k, a, b)
    b = run_sgcl_bounds(src, unroll=opts["unroll"], ctx=ctx)
    assert check_inside_enclosure(g, b) >= 5
