"""GPU parity of the hot kernel: the truncated N-D product (multivariate_taylor.rs:972-1012).

 * mid sizes: every kernel variant against the oracle on seeded dense tensors (distributions U and P of
   SURVEY 8d), ragged shapes, row subsets (the sharding primitive)
 * BASELINE sizes ((4,32) ... (6,16)): size-independent properties -- separable operands have a
   closed-form product (outer product of 1-D truncated convolutions), commutativity, linearity
"""
import numpy as np
import pytest

from helpers import RTOL, assert_bits, small_ints, synth_pgf, synth_uniform

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import genfer_b200
    c = genfer_b200.Context(0)
    genfer_b200.set_default_context(c)
    yield c
    genfer_b200.set_default_context(None)
    c.close()


def gpu_mul_raw(ctx, x, y, rshape, rows=None, fast=True, row_list=None):
    """Calls gtp_mul_rows_raw (rows = (begin, step, count), default all) or gtp_mul_rowlist_raw (row_list) through the
    C ABI on torch-owned device buffers."""
    import torch
    ctx.set_fast_mul(fast)
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    yd = torch.from_numpy(np.ascontiguousarray(y)).cuda()
    if rows is None:
        begin, step, count = 0, 1, rshape[0]
    else:
        begin, step, count = rows
    if row_list is not None:
        count = len(row_list)
    out = torch.full((count,) + tuple(rshape[1:]), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    if row_list is not None:
        ctx.mul_rowlist_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, row_list, out.data_ptr())
    else:
        ctx.mul_rows_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, begin, step, count, out.data_ptr())
    ctx.synchronize()
    ctx.set_fast_mul(1)
    return out.cpu().numpy()


def rel_err(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


CUBES = [(2, 16), (3, 16), (4, 8), (3, 32), (2, 32), (4, 12), (5, 8), (3, 24), (6, 4)]


@pytest.mark.parametrize("n,d", CUBES)
@pytest.mark.parametrize("dist", ["U", "P"])
def test_cube_product_matches_oracle(ctx, n, d, dist):
    from oracle import oracle as O
    gen = synth_uniform if dist == "U" else synth_pgf
    x, y = gen((d,) * n, 20230517), gen((d,) * n, 20231210)
    ref = O.mul_raw(x, y, (d,) * n)
    exact = gpu_mul_raw(ctx, x, y, (d,) * n, fast=False)
    assert np.array_equal(exact.view(np.uint64), ref.view(np.uint64)), "reference-order kernel must be bit-exact"
    fast = gpu_mul_raw(ctx, x, y, (d,) * n, fast=True)
    assert rel_err(fast, ref) <= RTOL, rel_err(fast, ref)   # all-positive inputs: no cancellation (SURVEY 8d)


RAGGED = [((3, 5), (4, 2), (6, 6)), ((3, 5), (4, 2), (5, 4)), ((1, 7), (6, 1), (6, 7)), ((4, 4, 4), (2, 1, 3), (5, 4, 6)),
          ((16, 16), (16, 16), (16, 9)), ((16, 16, 16), (5, 16, 16), (16, 16, 16)), ((9,), (5,), (11,)),
          ((2, 3, 4, 5), (5, 4, 3, 2), (6, 6, 6, 6)), ((8, 16), (16, 16), (16, 16))]


@pytest.mark.parametrize("xs,ys,rs", RAGGED)
def test_ragged_product_matches_oracle(ctx, xs, ys, rs):
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=False)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    got = gpu_mul_raw(ctx, x, y, rs, fast=True)
    np.testing.assert_allclose(got, ref, rtol=1e-11, atol=1e-12)


BLK_CUBES = [(4, 8), (4, 10), (4, 12), (4, 14), (4, 16), (3, 32), (3, 24), (4, 20), (3, 28), (3, 48), (4, 24), (5, 8), (5, 12)]


@pytest.mark.parametrize("n,d", BLK_CUBES)
@pytest.mark.parametrize("mode", [2, 18])
def test_blocked_kernel_cubes_match_oracle(ctx, n, d, mode):
    """The DFMA kernels on small cubes (mode 2 forces them; +16 switches the sliding 1x2 kernel off so the 2x2-blocked
    one runs everywhere): every chunk length 8..16, chunked last axes (20 = 2x10, 24 = 2x12, 28 = 2x14, 32 = 2x16,
    48 = 3x16), folded and unfolded b1."""
    from oracle import oracle as O
    x, y = synth_pgf((d,) * n, 20230517), synth_uniform((d,) * n, 20231210)
    ref = O.mul_raw(x, y, (d,) * n)
    got = gpu_mul_raw(ctx, x, y, (d,) * n, fast=mode)
    assert rel_err(got, ref) <= RTOL, rel_err(got, ref)


TILED_CUBES = [(4, 8, 34), (4, 12, 34), (4, 16, 34), (4, 16, 66), (4, 20, 34), (4, 24, 34), (4, 24, 66), (5, 8, 34), (5, 12, 34)]


@pytest.mark.parametrize("n,d,mode", TILED_CUBES)
def test_tiled_sliding_kernel_cubes_match_oracle(ctx, n, d, mode):
    """The sliding kernel with a tiled plane axis (mode 2 + 32: 4 planes per staged slab, + 64: 8 planes): interior tile
    pairs (cyclic plane classes) and the last tile sum (upper output planes masked), 120- and 96-thread CTAs."""
    from oracle import oracle as O
    x, y = synth_pgf((d,) * n, 20230517), synth_uniform((d,) * n, 20231210)
    ctx.set_fast_mul(mode)
    assert ctx.mul_kernel_kind((d,) * n, (d,) * n, (d,) * n) == 3
    ref = O.mul_raw(x, y, (d,) * n)
    got = gpu_mul_raw(ctx, x, y, (d,) * n, fast=mode)
    assert rel_err(got, ref) <= RTOL, rel_err(got, ref)


@pytest.mark.parametrize("mode", [2, 34])
def test_sliding_kernel_ragged_leading_axes(ctx, mode):
    """Operands whose leading (A) axes differ: the y strides are the y tensor's own."""
    from oracle import oracle as O
    xs, ys, rs = (5, 3, 8, 8, 8), (6, 4, 8, 8, 8), (8, 5, 8, 8, 8)
    rng = np.random.default_rng(11)
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ctx.set_fast_mul(mode)
    assert ctx.mul_kernel_kind(xs, ys, rs) == 3   # 8 untiled lanes are too few: both modes take the plane-tiled plan
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=mode)
    np.testing.assert_allclose(got, ref, rtol=1e-11, atol=1e-12)
    xs, ys, rs = (5, 3, 16, 16, 16), (6, 4, 16, 16, 16), (8, 5, 16, 16, 16)
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ctx.set_fast_mul(mode)
    assert ctx.mul_kernel_kind(xs, ys, rs) == 3
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=mode)
    np.testing.assert_allclose(got, ref, rtol=1e-11, atol=1e-12)


AXIS_CASES = [((282, 1), (282, 282), (282, 282)), ((1, 282), (282, 282), (282, 282)), ((247, 247), (36, 1), (247, 247)),
              ((161, 161), (1, 84), (161, 161)), ((40, 1, 1), (30, 20, 10), (50, 20, 10)), ((30, 20, 10), (1, 45, 1), (30, 40, 10)),
              ((1, 1, 300), (7, 5, 200), (7, 5, 260)), ((9, 200), (1, 300), (9, 499)), ((500,), (1,), (500,)), ((64, 64), (64, 1), (100, 64)),
              ((5, 1, 70, 1), (5, 3, 70, 9), (9, 3, 139, 9))]


@pytest.mark.parametrize("xs,ys,rs", AXIS_CASES)
def test_axis_convolution_kernel_is_bit_exact(ctx, xs, ys, rs):
    """1-d operand x N-d tensor (kernels_mul_axis.cu): bit-identical to the oracle's reference order, either operand order,
    axis first / middle / last, results shorter and longer than the operands."""
    from oracle import oracle as O
    rng = np.random.default_rng(sum(xs) + sum(ys))
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=True)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    ref = O.mul_raw(y, x, rs)
    got = gpu_mul_raw(ctx, y, x, rs, fast=True)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))


STENCIL_ROWS = [((97, 83, 91), (2, 1, 2), (98, 83, 92)), ((2, 1, 2), (97, 83, 91), (98, 83, 92)), ((120, 130, 75), (2, 2, 2), (121, 131, 76)),
                ((300, 1000), (3, 2), (300, 1001)), ((31, 29, 1, 33, 35), (2, 1, 1, 1, 2), (32, 29, 1, 33, 36)),
                ((97, 83, 91), (2, 1, 2), (90, 80, 91)), ((16,) * 6, (2, 1, 2, 1, 1, 2), (17, 16, 17, 16, 16, 17)),
                ((40, 9, 8, 7), (2, 1, 1, 3), (41, 9, 8, 9))]


@pytest.mark.parametrize("xs,ys,rs", STENCIL_ROWS)
def test_row_staged_small_operand_product_is_bit_exact(ctx, xs, ys, rs):
    """The row-staged bulk-copy (TMA) kernel of the fused Horner loop (k_horner_rows), driven as a single product: same
    bits as the reference order, either operand order, truncated results, unit axes, odd row lengths, merged row blocks."""
    from oracle import oracle as O
    rng = np.random.default_rng(sum(rs))
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=1 + 32768)     # the row-staged kernel (opt-in for single products)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    got = gpu_mul_raw(ctx, x, y, rs, fast=True)          # default: the gather kernels give the same bits
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))


ODD_SHAPES = [((27,) * 3,) * 3, ((13,) * 4,) * 3, ((17,) * 4,) * 3, ((31,) * 3,) * 3, ((9,) * 5,) * 3,
              ((13, 17, 19, 21), (11, 17, 15, 21), (13, 17, 19, 21)), ((5, 27, 27, 27), (3, 20, 27, 25), (7, 27, 27, 27))]


@pytest.mark.parametrize("xs,ys,rs", ODD_SHAPES)
def test_odd_shaped_products_leave_the_reference_order_kernel(ctx, xs, ys, rs):
    """Cube edges 27, 31, 17 ... (limit + 1 + sum of orders): zero-extended to the DFMA kernels' extents and cropped --
    1e-12 against the oracle (all-positive inputs), and no longer on the ~0.15 TFLOP/s reference-order kernel."""
    from oracle import oracle as O
    from helpers import synth_uniform
    x, y = synth_uniform(xs, 101), synth_uniform(ys, 202)
    assert ctx.mul_kernel_kind(xs, ys, rs) in (2, 3, 6, 7)
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=True)
    assert rel_err(got, ref) <= RTOL, rel_err(got, ref)
    rows = (1, 2, (rs[0] - 1) // 2)                       # a cyclic row shard goes through the same plan
    got_rows = gpu_mul_raw(ctx, x, y, rs, rows=rows, fast=True)
    assert rel_err(got_rows, ref[rows[0]::rows[1]][:rows[2]]) <= RTOL


@pytest.mark.parametrize("n,d", [(4, 12), (4, 16), (5, 12), (5, 16), (4, 8), (4, 24), (4, 10)])
def test_kernel_selection(ctx, n, d):
    """Dense cube slabs take the sliding kernel (3): whole slabs when they give >= 16 folded lanes and fit in shared
    memory, plane-tiled otherwise; rows not divisible by 4 go to the blocked kernel (2)."""
    ctx.set_fast_mul(2)
    kind = ctx.mul_kernel_kind((d,) * n, (d,) * n, (d,) * n)
    ctx.set_fast_mul(1)
    assert kind == (2 if d == 10 else 3)


BLK_RAGGED = [((5, 7, 9, 16), (6, 4, 9, 16), (8, 9, 12, 16)), ((3, 5, 16), (4, 2, 16), (6, 6, 16)),
              ((4, 4, 5, 24), (2, 3, 7, 24), (5, 4, 9, 24)), ((16, 16, 1, 8), (16, 1, 16, 8), (16, 16, 16, 8)),
              ((7, 3, 12), (7, 5, 12), (7, 7, 12)), ((2, 9, 9, 32), (3, 9, 9, 32), (4, 9, 5, 32)),
              ((6, 1, 1, 10), (6, 1, 1, 10), (6, 1, 1, 10))]


@pytest.mark.parametrize("xs,ys,rs", BLK_RAGGED)
def test_blocked_kernel_ragged_match_oracle(ctx, xs, ys, rs):
    """Odd row counts (zero-filled pair rows), result shorter / longer than the operands, unit axes."""
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=2)
    np.testing.assert_allclose(got, ref, rtol=1e-11, atol=1e-12)


BLK_ROW_SHAPES = [((12,) * 4,) * 3,                                   # folded item table (dense cube slabs)
                  ((16,) * 3,) * 3,                                   # evenly dealt table (single-plane slabs)
                  ((5, 7, 9, 16), (6, 4, 9, 16), (8, 9, 12, 16))]     # evenly dealt, odd row counts, unequal boxes


@pytest.mark.parametrize("xs,ys,rs", BLK_ROW_SHAPES)
def test_blocked_kernel_row_shards_are_exact(ctx, xs, ys, rs):
    """Row shards through the 2x2-blocked kernel (mode 18 forces the DFMA kernels and switches the sliding one off), as
    partitioned multi-GPU products send them: cyclic rows (gtp_mul_rows_raw) and a folded-cyclic row list
    (gtp_mul_rowlist_raw).  Small-integer operands: bit for bit against the oracle."""
    from oracle import oracle as O
    from genfer_b200.partition import rows_for_rank
    x, y = small_ints(xs, 61), small_ints(ys, 62)
    ref = O.mul_raw(x, y, rs)
    ctx.set_fast_mul(18)
    kind = ctx.mul_kernel_kind(xs, ys, rs)
    ctx.set_fast_mul(1)
    assert kind == 2
    cyclic = (1, 3, len(range(1, rs[0], 3)))
    assert_bits(gpu_mul_raw(ctx, x, y, rs, rows=cyclic, fast=18), ref[1::3])
    folded = rows_for_rank(rs[0], 2, 1)
    assert_bits(gpu_mul_raw(ctx, x, y, rs, row_list=folded, fast=18), ref[folded])


@pytest.mark.parametrize("n,d,world", [(3, 16, 2), (4, 8, 4), (3, 16, 8), (4, 16, 8)])
def test_row_shards_tile_the_product(ctx, n, d, world):
    """Cyclic leading-axis shards (SURVEY 8e) computed independently reassemble the full product."""
    x, y = synth_uniform((d,) * n, 1), synth_uniform((d,) * n, 2)
    full = gpu_mul_raw(ctx, x, y, (d,) * n)
    out = np.empty_like(full)
    for r in range(world):
        cnt = len(range(r, d, world))
        out[r::world] = gpu_mul_raw(ctx, x, y, (d,) * n, rows=(r, world, cnt))
    # partial rows meet in HBM through RED.ADD and the units of a row subset split the j box differently from those of the
    # full product, so shards agree with the full launch to rounding, not bit for bit (the reference-order kernel does)
    assert rel_err(out, full) <= 1e-13
    ctx.set_fast_mul(0)
    full0 = gpu_mul_raw(ctx, x, y, (d,) * n, fast=False)
    out0 = np.empty_like(full0)
    for r in range(world):
        cnt = len(range(r, d, world))
        out0[r::world] = gpu_mul_raw(ctx, x, y, (d,) * n, rows=(r, world, cnt), fast=False)
    assert np.array_equal(out0.view(np.uint64), full0.view(np.uint64))


def conv1d_trunc(a, b, n):
    return np.convolve(a, b)[:n]


@pytest.mark.parametrize("n,d", [(4, 32), (5, 16), (6, 12), (5, 24), (6, 16)])
def test_baseline_sizes_separable_closed_form(ctx, n, d):
    """At BASELINE's sizes: X = (x)_a, Y = (y)_a outer products  =>  X*Y = outer product of the 1-D truncated
    convolutions.  Checks every coefficient of the full-size product without a CPU N-D reference."""
    import torch
    rng = np.random.default_rng(n * 100 + d)
    xa = [rng.uniform(0.5, 1.5, d) for _ in range(n)]
    ya = [rng.uniform(0.5, 1.5, d) for _ in range(n)]

    def outer(vs):
        t = torch.ones((), dtype=torch.float64, device="cuda")
        for v in vs:
            t = t.unsqueeze(-1) * torch.from_numpy(v).cuda()
        return t.contiguous()
    X, Y = outer(xa), outer(ya)
    Z = torch.empty_like(X)
    torch.cuda.synchronize()
    ctx.mul_rows_raw(X.shape, X.data_ptr(), Y.shape, Y.data_ptr(), X.shape, 0, 1, d, Z.data_ptr())
    ctx.synchronize()
    expect = outer([conv1d_trunc(xa[i], ya[i], d) for i in range(n)])
    err = torch.max(torch.abs(Z - expect) / expect).item()
    assert err <= 1e-12, err
    # commutativity on the same operands
    Z2 = torch.empty_like(X)
    ctx.mul_rows_raw(Y.shape, Y.data_ptr(), X.shape, X.data_ptr(), X.shape, 0, 1, d, Z2.data_ptr())
    ctx.synchronize()
    assert torch.max(torch.abs(Z2 - Z) / Z).item() <= 1e-12


def test_operator_level_product_uses_fast_kernel(ctx):
    """TaylorPoly * TaylorPoly on dense cubes goes through the full dispatch into the tiled kernel."""
    import genfer_b200
    from oracle import oracle as O
    d, n = 16, 3
    x, y = synth_pgf((d,) * n, 5), synth_pgf((d,) * n, 6)
    g = genfer_b200.taylor(x) * genfer_b200.taylor(y)
    o = O.taylor(x) * O.taylor(y)
    assert g.array_shape() == o.array_shape() and g.shape() == o.shape()
    assert rel_err(g.array(), o.array()) <= RTOL


STENCIL = [((40, 30, 40), (2, 1, 2), (41, 30, 41)), ((2, 1, 2), (40, 30, 40), (41, 30, 41)), ((40, 30, 40), (2, 1, 2), (40, 30, 40)),
           ((64, 80), (3, 2), (66, 81)), ((64, 80), (3, 2), (50, 81)), ((5000,), (7,), (5006,)), ((7,), (5000,), (4000,)),
           ((20, 20, 20), (1, 3, 1), (20, 22, 20)), ((9, 1, 30, 1, 25), (2, 1, 2, 1, 3), (10, 1, 31, 1, 27)),
           ((16, 16, 16, 4), (2, 2, 2, 2), (17, 17, 17, 5)), ((300, 40), (1, 32), (300, 71)), ((70, 1, 70), (4, 1, 8), (73, 1, 77))]


@pytest.mark.parametrize("xs,ys,rs", STENCIL)
def test_stencil_product_bit_exact(ctx, xs, ys, rs):
    """Products with one operand of at most 32 coefficients (multilinear substitutions, thinning factors) take the
    HBM-bound stencil kernel; it visits the terms in the reference's order, so it is bit-identical to the oracle --
    either operand small, truncated results, unit axes, signed zeros, and leading-axis row subsets."""
    from oracle import oracle as O
    rng = np.random.default_rng(sum(xs) + 7 * sum(ys))
    x, y = rng.standard_normal(xs), rng.standard_normal(ys)
    x.flat[rng.integers(0, x.size, max(1, x.size // 11))] = -0.0
    y.flat[rng.integers(0, y.size, max(1, y.size // 5))] = 0.0
    ref = O.mul_raw(x, y, rs)
    got = gpu_mul_raw(ctx, x, y, rs, fast=True)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    off = gpu_mul_raw(ctx, x, y, rs, fast=257)       # + 256: stencil kernel off -> reference-order kernel
    assert np.array_equal(off.view(np.uint64), ref.view(np.uint64))
    one = gpu_mul_raw(ctx, x, y, rs, fast=513)       # + 512: one coefficient per thread instead of four
    assert np.array_equal(one.view(np.uint64), ref.view(np.uint64))
    if rs[0] > 3:
        cnt = len(range(1, rs[0], 3))
        rows = gpu_mul_raw(ctx, x, y, rs, rows=(1, 3, cnt), fast=True)
        assert np.array_equal(rows.view(np.uint64), ref[1::3].view(np.uint64))
