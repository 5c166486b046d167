"""A/B timing of the sliding product kernel on whole 16^3 slabs: the run-granular kernel (k_mul_slide16, default) against
the step-table kernel (gtp_ctx_set_fast_mul bit 1 << 19).  CUDA events around `--reps` back-to-back products per
measurement; the two paths alternate for `--rounds` rounds on the same operands, so drifting clocks hit both alike.
Operands are 128 MiB (6 x 16) and 8 MiB (5 x 16); both products are FP64-pipe bound, not bandwidth bound.

usage: ab_slide.py [--rounds R] [--reps K] [--out FILE.json] [NxD ...]      (default 6x16 5x16)
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import genfer_b200  # noqa: E402

SLIDE_TABLE = 1 << 19
PATHS = {"runs": 1, "table": 1 | SLIDE_TABLE}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (f.strip() for f in out.split(","))))
    except Exception as e:   # the timings stand without it
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=0, help="products per measurement (0: 4 for 6x16, 40 for smaller)")
    ap.add_argument("--out")
    ap.add_argument("workloads", nargs="*", default=["6x16", "5x16"])
    args = ap.parse_args()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = genfer_b200.Context(0, stream=stream.cuda_stream)
    res = {"gpu_before": gpu_info(), "rounds": args.rounds, "workloads": []}
    for w in args.workloads:
        n, d = (int(t) for t in w.split("x"))
        shape = (d,) * n
        g = torch.Generator(device="cuda").manual_seed(1)
        x = torch.rand(shape, dtype=torch.float64, device="cuda", generator=g)
        y = torch.rand(shape, dtype=torch.float64, device="cuda", generator=g)
        z = {p: torch.empty(shape, dtype=torch.float64, device="cuda") for p in PATHS}
        macs = genfer_b200.mul_macs(shape, shape, shape)
        reps = args.reps or (4 if macs > 1e12 else 40)

        def run(path):
            ctx.set_fast_mul(PATHS[path])
            ctx.mul_rows_raw(shape, x.data_ptr(), shape, y.data_ptr(), shape, 0, 1, d, z[path].data_ptr())

        kinds = {}
        for p in PATHS:   # warm-up: plan build, module load, clocks
            ctx.set_fast_mul(PATHS[p])
            kinds[p] = ctx.mul_kernel_kind(shape, shape, shape)
            for _ in range(2):
                run(p)
        torch.cuda.synchronize()
        ms = {p: [] for p in PATHS}
        for r in range(args.rounds):
            for p in (PATHS if r % 2 == 0 else reversed(list(PATHS))):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    run(p)
                e1.record()
                torch.cuda.synchronize()
                ms[p].append(e0.elapsed_time(e1) / reps)
        ctx.set_fast_mul(1)
        a, b = z["runs"], z["table"]
        rel = float(((a - b).abs() / b.abs()).max())
        rec = {"workload": w, "macs": macs, "reps_per_measurement": reps, "kernel_kind": kinds, "max_rel_diff": rel}
        for p in PATHS:
            rec[p] = {"ms": ms[p], "ms_min": min(ms[p]), "ms_max": max(ms[p]),
                      "tflops_best": 2 * macs / min(ms[p]) / 1e9}
        rec["speedup_best"] = min(ms["table"]) / min(ms["runs"])
        rec["speedup_conservative"] = min(ms["table"]) / max(ms["runs"])   # slowest new-path run against the fastest table run
        res["workloads"].append(rec)
        print(json.dumps(rec), flush=True)
        del x, y, z
    res["gpu_after"] = gpu_info()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"gpu_before": res["gpu_before"], "gpu_after": res["gpu_after"]}), flush=True)


if __name__ == "__main__":
    main()
