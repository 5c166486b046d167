"""Shared helpers for the parity tests: oracle <-> device comparison."""
import numpy as np

from oracle import oracle as O

RTOL = 1e-12  # north_star: results within 1e-12 relative of the reference f64 path


def to_oracle(a, degrees=None):
    a = np.asarray(a, dtype=np.float64)
    return O.TaylorPoly.new(a, a.shape if degrees is None else degrees)


def assert_meta_equal(g, o):
    """Integer work must be bit-exact: stored shape and degrees_p1."""
    assert g.array_shape() == o.array_shape(), (g.array_shape(), o.array_shape())
    assert g.shape() == o.shape(), (g.shape(), o.shape())


def assert_same(g, o):
    """Bit-exact agreement (shape, degrees and every coefficient incl. signed zeros / NaN patterns)."""
    assert_meta_equal(g, o)
    ga, oa = g.array(), o.array()
    assert np.array_equal(ga.view(np.uint64), oa.view(np.uint64)), f"\n gpu={ga}\n ref={oa}"


def assert_close(g, o, rtol=RTOL, atol_scale=None):
    """|gpu - ref| <= rtol * max(|ref|, floor): floor = rtol * max|ref| guards entries that are exact
    zeros in the reference but tiny non-zeros after FMA/re-ordering (SURVEY 7 'parity budget')."""
    assert_meta_equal(g, o)
    ga, oa = g.array(), o.array()
    scale = np.max(np.abs(oa)) if oa.size else 0.0
    floor = (atol_scale if atol_scale is not None else scale) * rtol
    err = np.abs(ga - oa)
    bound = rtol * np.abs(oa) + floor
    bad = ~(err <= bound) & ~(np.isnan(ga) & np.isnan(oa)) & ~((ga == oa))
    assert not bad.any(), f"max rel err {np.max(err / np.maximum(np.abs(oa), 1e-300))}\n gpu={ga}\n ref={oa}"


def small_ints(shape, seed):
    """Operands of integers 0..3: every product and partial sum of a DFMA product kernel is then an exact integer in f64,
    whatever the summation or RED.ADD meeting order, so a missed or repeated multiply-add shows as a bit difference."""
    return np.random.default_rng(seed).integers(0, 4, size=shape).astype(np.float64)


def assert_bits(got, ref):
    diff = np.flatnonzero(got.view(np.uint64) != ref.view(np.uint64))
    assert diff.size == 0, f"{diff.size} coefficients differ, first at flat {diff[0]}: {got.flat[diff[0]]} != {ref.flat[diff[0]]}"


from genfer_b200.synth import splitmix64, synth_pgf, synth_uniform  # noqa: E402,F401


# ---------------------------------------------------------------------------------------------
# north_star check 2, end to end: f64 results inside the Interval<F64> enclosure of the same evaluation
# ---------------------------------------------------------------------------------------------
# programs whose Interval<F64> evaluation takes more than a few seconds on one host core: left out of the CPU suite (kept to a
# few minutes); the GPU suite (-m gpu) checks the BASELINE programs among them too (ENCLOSURE_GPU_EXTRA: 20-60 s of oracle each)
ENCLOSURE_GPU_EXTRA = ("real_world/population2000.sgcl", "real_world/population_modified2000.sgcl", "real_world/population_2000_1vars.sgcl",
                       "real_world/switchpoint.sgcl", "real_world/cont_switchpoint.sgcl", "real_world/hmm.sgcl", "slow/two_populations2000.sgcl")
ENCLOSURE_SLOW = {"mixture", "hmm", "switchpoint", "cont_switchpoint", "two_populations2000", "two_populations", "nested_infer_expensive",
                  "population_modified2000", "population2000", "population_2000_1vars", "population", "population_modified"}


def check_inside_enclosure(result, bounds):
    """`result`: the f64 run (oracle or GPU; .total, .mean, .raw2.., .probs); `bounds`: oracle.run_sgcl_bounds of the same
    program.  Z and the raw moments are compared where the report's post-processing is the identity (no rest mass, Z
    inside [0, 1]); a probability that the report clamped to 0 or 1, or to which it added the rest mass, is compared
    with the correspondingly relaxed interval.  Returns the number of quantities checked."""
    import math
    checked = 0
    rest_lo, rest_hi = bounds.rest
    no_rest = rest_lo == 0.0 and rest_hi == 0.0
    finite = all(math.isfinite(x) for x in bounds.total)
    if no_rest and finite and 0.0 <= bounds.total[0] and bounds.total[1] <= 1.0:
        assert bounds.total[0] <= result.total <= bounds.total[1], ("Z", result.total, bounds.total)
        checked += 1
        for name, value, (lo, hi) in zip(("E", "raw2", "raw3", "raw4"), (result.mean, result.raw2, result.raw3, result.raw4),
                                         bounds.raw_moments):
            if math.isfinite(lo) and math.isfinite(hi) and lo >= 0.0:
                assert lo <= value <= hi, (name, value, (lo, hi))
                checked += 1
    for i, (p, (lo, hi)) in enumerate(zip(result.probs, bounds.probs)):
        if not (math.isfinite(lo) and math.isfinite(hi)):
            continue
        lo_c, hi_c = max(lo, 0.0), min(hi + max(rest_hi, 0.0), 1.0)    # clamping to [0, 1] and `p + rest` in the report
        assert min(lo_c, 1.0) <= p <= max(hi_c, 0.0), (f"p({i})", p, (lo, hi), bounds.rest)
        checked += 1
    return checked
