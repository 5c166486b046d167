"""Times the symbolic mode (`-s`) and univariate programs on the GPU; one JSON line per measurement.

- per `tests/golden/sgcl_symbolic` fixture: best-of-N wall time of run_sgcl(symbolic=True), its launches (also without
  GenFun::simplify, i.e. the symbolic evaluation alone), whether the report equals the `.expect` byte for byte, and the
  oracle's best-of-N time on one host core;
- per random DAG of tests/test_gpu_uni_program.py: the per-op replay through gtu_* against recording + one program run
  (and the run alone), alternated in the same process, with the DAG's level count and widest level.
The first line names the card and its power limit.
usage: time_symbolic.py [--reps N] [--out FILE]"""
import argparse
import glob
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import genfer_b200  # noqa: E402
from oracle import oracle as O  # noqa: E402
import test_gpu_uni_program as T  # noqa: E402  (the random DAGs and both evaluation paths)


def best(f, reps):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t)
    return min(ts)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the timing is still worth having; say what is missing
        return {"gpu": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    ctx = genfer_b200.Context(0)
    emit(dict(card(), what="device", host_cores_for_oracle=1))
    cpus = os.sched_getaffinity(0)
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "sgcl_symbolic", "*.sgcl"))):
        src = open(path).read()
        expect = open(path[:-5] + ".expect").read()
        kw = T.flags_of(src)
        g = genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **kw)   # warm-up
        l0 = ctx.launch_count
        g = genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **kw)
        launches = ctx.launch_count - l0
        l0 = ctx.launch_count
        genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **dict(kw, no_simplify_gf=True))
        eval_launches = ctx.launch_count - l0
        t_gpu = best(lambda: genfer_b200.run_sgcl(src, ctx=ctx, symbolic=True, **kw), a.reps)
        os.sched_setaffinity(0, {min(cpus)})
        try:
            O.run_sgcl(src, symbolic=True, **kw)
            t_cpu = best(lambda: O.run_sgcl(src, symbolic=True, **kw), a.reps)
        finally:
            os.sched_setaffinity(0, cpus)
        emit({"what": "fixture", "program": os.path.relpath(path, ROOT), "gpu_ms": round(t_gpu * 1e3, 4), "launches": launches,
              "launches_without_simplify": eval_launches,
              "nodes_evaluated": g.nodes_evaluated, "byte_identical": g.report == expect, "oracle_1core_ms": round(t_cpu * 1e3, 4)})

    G = (genfer_b200, ctx)
    for seed, top in T.DAG_SEEDS:
        nodes = T.random_dag(seed, top=top)
        levels, width = T.dag_shape(nodes)
        n_ops = sum(1 for n in nodes if n[0] not in ("const", "coeffs"))

        def per_op():
            vals = T.eval_per_op(G, nodes)
            ctx.synchronize()
            return vals

        def program():
            p, slots = T.record(G, nodes)
            return p.run(*slots)

        per_op(), program()   # warm-up
        p, slots = T.record(G, nodes)
        t_op, t_prog, t_run = [], [], []
        for _ in range(a.reps):   # alternated
            t_op.append(best(per_op, 1))
            t_prog.append(best(program, 1))
            t_run.append(best(lambda: p.run(*slots), 1))
        ref = [v.coeffs() for v in per_op()]
        got = program()
        try:
            for r, g_ in zip(ref, got):
                T.assert_bits(g_, r)
            same = True
        except AssertionError:
            same = False
        emit({"what": "random_dag", "seed": seed, "top_order": top, "ops": n_ops, "levels": levels, "max_level_width": width,
              "per_op_ms": round(min(t_op) * 1e3, 4), "record_and_run_ms": round(min(t_prog) * 1e3, 4),
              "run_ms": round(min(t_run) * 1e3, 4), "bit_identical": same})
    ctx.close()


if __name__ == "__main__":
    main()
