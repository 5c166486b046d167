"""The product kind reported by gtp_mul_kernel_kind (what bench.py prints as "kernel") is the kernel that runs.

Every whole-result product of the corpus runs in a fresh context of one child process with GTP_LAUNCH_HIST=1; the launch
census printed when the context closes must show the kernels its kind names: 3 the sliding DFMA kernel, 2 the blocked one,
6 / 7 a zero-extending copy and then the blocked / sliding kernel, 0 neither DFMA kernel.
"""
import os
import re
import subprocess
import sys

import pytest

from test_gpu_product import (AXIS_CASES, BLK_RAGGED, BLK_ROW_SHAPES, CUBES, ODD_SHAPES, RAGGED, STENCIL, STENCIL_ROWS,
                              TILED_CUBES)

pytestmark = pytest.mark.gpu

# test_gpu_product.py's shapes, and bench.py's headline and sweep cubes
CORPUS = sorted({tuple(map(tuple, c)) for c in
                 RAGGED + AXIS_CASES + STENCIL_ROWS + ODD_SHAPES + BLK_RAGGED + BLK_ROW_SHAPES + STENCIL
                 + [((d,) * n,) * 3 for n, d in CUBES + [(n, d) for n, d, _ in TILED_CUBES]]
                 + [((5, 3, 8, 8, 8), (6, 4, 8, 8, 8), (8, 5, 8, 8, 8)), ((5, 3, 16, 16, 16), (6, 4, 16, 16, 16), (8, 5, 16, 16, 16))]
                 + [((d,) * n,) * 3 for n, d in ((6, 16), (4, 32), (5, 16), (6, 12), (5, 24), (4, 27), (4, 31), (5, 17))]})

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


@pytest.fixture(scope="module")
def launched():
    """{(xs, ys, rs): (kind, set of kernel names in the product's launch census)}"""
    env = dict(os.environ, GTP_LAUNCH_HIST="1")
    env.pop("GTP_FAST_MUL", None)
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", CHILD, repr(CORPUS)], cwd=repo, env=env, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    out = {}
    for part in r.stderr.split("@@product ")[1:]:
        i = int(part.split("\n", 1)[0])
        kind = int(re.search(r"^@@kind (\d+)$", part, re.M).group(1))
        names = set(re.findall(r"^\[gtp launches\]\s+\d+\s+(.+)$", part, re.M))
        out[CORPUS[i]] = (kind, names)
    assert len(out) == len(CORPUS)
    return out


@pytest.mark.parametrize("xs,ys,rs", CORPUS, ids=lambda s: "x".join(map(str, s)))
def test_reported_kind_is_the_kernel_that_runs(launched, xs, ys, rs):
    kind, names = launched[(xs, ys, rs)]
    slide = any("k_mul_slide" in n for n in names)
    blk = any("k_mul_blk" in n for n in names)
    copy = any("k_ew" in n for n in names)
    if kind == 3:
        assert slide and not blk, names
    elif kind == 2:
        assert blk and not slide, names
    elif kind == 7:
        assert slide and not blk and copy, names
    elif kind == 6:
        assert blk and not slide and copy, names
    else:
        assert kind == 0 and not slide and not blk, (kind, names)
