"""Timing of products on 9+ non-unit axes -- the fastest applicable route (the trailing-box DFMA kernel k_mul_box, or the
zero-extended blocked kernel) against the reference-order kernel k_mul_ordered<NE> -- and of an end-to-end program with nine
live variables, against the CPU oracle.  One JSON line per measurement on stdout; the first line names the card and
its power limit.  usage: time_high_rank.py [--program path.sgcl]"""
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np
import torch
import genfer_b200
from oracle import oracle as O

SHAPES = [(4,) * 10, (3,) * 12, (4,) * 9, (6,) * 9, (8,) + (3,) * 9]
PROGRAM = os.path.join(REPO, "tests", "thinning_tree_9vars.sgcl")


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def main():
    program = sys.argv[sys.argv.index("--program") + 1] if "--program" in sys.argv else PROGRAM
    emit(card=card(), torch=torch.__version__)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = genfer_b200.Context(0, stream=stream.cuda_stream)
    peak, _ = ctx.fp64_peak_probe(0)
    emit(probe="dfma", tflops=round(peak / 1e12, 2))
    for shape in SHAPES:
        macs = genfer_b200.mul_macs(shape, shape, shape)
        x = torch.rand(shape, dtype=torch.float64, device="cuda")
        y = torch.rand(shape, dtype=torch.float64, device="cuda")
        z = torch.empty(shape, dtype=torch.float64, device="cuda")

        def run():
            ctx.mul_rows_raw(shape, x.data_ptr(), shape, y.data_ptr(), shape, 0, 1, shape[0], z.data_ptr())

        # the oracle's leading-axis row 0 (the cheapest row), where that costs at most 2e9 MACs: parity and the CPU rate
        row0 = genfer_b200.mul_macs((1,) + shape[1:], (1,) + shape[1:], (1,) + shape[1:])
        ref = cpu_gmacs = None
        if row0 <= 2e9:
            t0 = time.perf_counter()
            ref, cpu_macs = O.mul_rows(x.cpu().numpy(), y.cpu().numpy(), shape, [0])
            cpu_gmacs = round(cpu_macs / (time.perf_counter() - t0) / 1e9, 3)
        ms_by_mode = {}
        for mode in (1, 0):   # the fastest applicable route, then the reference-order kernel alone
            ctx.set_fast_mul(mode)
            run()   # warm-up: module load, plan build
            ctx.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run()
            e1.record(stream)
            e1.synchronize()
            one = e0.elapsed_time(e1)
            reps = max(1, min(20, int(1000.0 / max(one, 1e-3))))   # about one second of work
            e0.record(stream)
            for _ in range(reps):
                run()
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / reps
            ms_by_mode[mode] = ms
            tflops = 2 * macs / (ms * 1e-3) / 1e12
            err = None
            if ref is not None:
                got = z[0].cpu().numpy()
                err = float(np.max(np.abs(got - ref[0]) / np.maximum(np.abs(ref[0]), 1e-300)))
            emit(shape=list(shape), fast_mul=mode, kind=ctx.mul_kernel_kind(shape, shape, shape), macs=macs, ms=round(ms, 3),
                 reps=reps, tflops=round(tflops, 4), of_dfma_probe=round(tflops * 1e12 / peak, 5), cpu_oracle_gmacs=cpu_gmacs,
                 row0_max_rel_err=err)
        ctx.set_fast_mul(1)
        emit(shape=list(shape), reference_order_over_fastest=round(ms_by_mode[0] / ms_by_mode[1], 2))
        del x, y, z
    ctx.close()
    # end to end: the program on the device (second run timed: the first loads modules) and on the CPU oracle
    src = open(program).read()
    opts = genfer_b200.parse_flags(src)
    ctx = genfer_b200.Context(0)
    genfer_b200.run_sgcl(src, limit=opts["limit"], no_probs=opts["no_probs"], ctx=ctx)
    times = []
    for _ in range(9):   # host clock around a whole run (it ends with the report read back); median of 9
        t0 = time.perf_counter()
        g = genfer_b200.run_sgcl(src, limit=opts["limit"], no_probs=opts["no_probs"], ctx=ctx)
        times.append(time.perf_counter() - t0)
    gpu_s = float(np.median(times))
    ctx.close()
    t0 = time.perf_counter()
    o = O.run_sgcl(src, limit=opts["limit"], no_probs=opts["no_probs"])
    cpu_s = time.perf_counter() - t0
    emit(program=os.path.relpath(program, REPO), gpu_s_median_of_9=round(gpu_s, 5), gpu_s_min=round(min(times), 5), cpu_oracle_s=round(cpu_s, 4),
         report_identical=g.report == o.report, Z=g.total, Z_oracle=o.total)


if __name__ == "__main__":
    main()
