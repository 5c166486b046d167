"""The run-granular sliding kernel (k_mul_slide16: whole 16^3 slabs) against the oracle and against the step-table kernel.

Operands of small integers (0..3) make every product and every partial sum an exact integer in f64, whatever the
summation order or the RED.ADD meeting order: a multiply-add that the schedule misses or repeats shows up as a bit
difference, not as a rounding-level one.  Each case runs both kernels (fast_mul 1: default, 1 | SLIDE_TABLE: the
step-table kernel) and requires both to be bit-identical to the oracle.
"""
import numpy as np
import pytest

from helpers import assert_bits, small_ints

pytestmark = pytest.mark.gpu

SLIDE_TABLE = 1 << 19   # gtp_ctx_set_fast_mul bit: whole 16^3 slabs on the step-table kernel
MODES = [1, 1 | SLIDE_TABLE]
CUBE5 = (16,) * 5
ROWS5_CYCLIC = (2, 4, 3)   # row_begin, row_step, row_count: rows 2, 6, 10
ROWS5_FOLDED = [3, 12]     # rank 3 of 8 (partition.rows_for_rank)


@pytest.fixture(scope="module")
def ctx():
    import genfer_b200
    c = genfer_b200.Context(0)
    genfer_b200.set_default_context(c)
    yield c
    genfer_b200.set_default_context(None)
    c.close()


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
        assert ctx.mul_kernel_kind(x.shape, y.shape, rshape) == 3
        if row_list is not None:
            ctx.mul_rowlist_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, row_list, out.data_ptr())
        else:
            begin, step, n = rows if rows else (0, 1, rshape[0])
            ctx.mul_rows_raw(x.shape, xd.data_ptr(), y.shape, yd.data_ptr(), rshape, begin, step, n, out.data_ptr())
        ctx.synchronize()
    finally:
        ctx.set_fast_mul(1)
    return out.cpu().numpy()


@pytest.fixture(scope="module")
def cube5():
    """5 x 16 integer operands and the oracle's rows 2, 3, 6, 10, 12 (the only rows the 5 x 16 cases compare)."""
    from oracle import oracle as O
    x, y = small_ints(CUBE5, 51), small_ints(CUBE5, 52)
    rows = sorted({*range(ROWS5_CYCLIC[0], ROWS5_CYCLIC[0] + ROWS5_CYCLIC[1] * ROWS5_CYCLIC[2], ROWS5_CYCLIC[1]), *ROWS5_FOLDED})
    ref, _ = O.mul_rows(x, y, CUBE5, rows)
    return x, y, ref


@pytest.mark.parametrize("mode", MODES)
def test_exact_4x16(ctx, mode):
    from oracle import oracle as O
    shape = (16,) * 4
    x, y = small_ints(shape, 41), small_ints(shape, 42)
    assert_bits(device_product(ctx, mode, x, y, shape), O.mul_raw(x, y, shape))


@pytest.mark.parametrize("mode", MODES)
def test_exact_5x16_cyclic_rows(ctx, cube5, mode):
    x, y, ref = cube5
    begin, step, n = ROWS5_CYCLIC
    got = device_product(ctx, mode, x, y, CUBE5, rows=ROWS5_CYCLIC)
    assert_bits(got, ref[begin:begin + step * n:step])


@pytest.mark.parametrize("mode", MODES)
def test_exact_5x16_folded_cyclic_rows(ctx, cube5, mode):
    x, y, ref = cube5
    assert_bits(device_product(ctx, mode, x, y, CUBE5, row_list=ROWS5_FOLDED), ref[ROWS5_FOLDED])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_exact_4x16_folded_cyclic_rows_every_rank(ctx, mode, world):
    from oracle import oracle as O
    from genfer_b200.partition import rows_for_rank
    shape = (16,) * 4
    x, y = small_ints(shape, 43), small_ints(shape, 44)
    ref = O.mul_raw(x, y, shape)
    for rank in range(world):
        rows = rows_for_rank(16, world, rank)
        assert_bits(device_product(ctx, mode, x, y, shape, row_list=rows), ref[rows])


UNEQUAL = [((5, 3, 16, 16, 16), (6, 4, 16, 16, 16), (8, 5, 16, 16, 16)),
           ((7, 16, 16, 16), (12, 16, 16, 16), (16, 16, 16, 16)),
           ((2, 9, 16, 16, 16), (3, 5, 16, 16, 16), (3, 11, 16, 16, 16))]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("xs,ys,rs", UNEQUAL)
def test_exact_unequal_leading_axes(ctx, mode, xs, ys, rs):
    """Leading axes of different extent in x, y and the result (the y strides are y's own), 16^3 slabs."""
    from oracle import oracle as O
    x, y = small_ints(xs, 45), small_ints(ys, 46)
    assert_bits(device_product(ctx, mode, x, y, rs), O.mul_raw(x, y, rs))


def test_6x16_matches_step_table_kernel(ctx):
    """The headline product (uniform [0, 1) operands, every one of the 16.8 M coefficients): run-granular kernel against
    the step-table kernel at relative 1e-12 (the two sum in different orders)."""
    import torch
    from genfer_b200.synth import SEED_X, SEED_Y, synth_uniform
    shape = (16,) * 6
    xd = torch.from_numpy(synth_uniform(shape, SEED_X)).cuda()
    yd = torch.from_numpy(synth_uniform(shape, SEED_Y)).cuda()
    outs = []
    for mode in MODES:
        out = torch.full(shape, float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ctx.set_fast_mul(mode)
        try:
            assert ctx.mul_kernel_kind(shape, shape, shape) == 3
            ctx.mul_rows_raw(shape, xd.data_ptr(), shape, yd.data_ptr(), shape, 0, 1, 16, out.data_ptr())
            ctx.synchronize()
        finally:
            ctx.set_fast_mul(1)
        outs.append(out)
    new, table = outs
    assert bool(torch.isfinite(new).all()) and bool((table > 0).all())
    rel = float(((new - table).abs() / table).max())
    assert rel <= 1e-12, rel
