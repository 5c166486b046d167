#!/usr/bin/env python
"""bench.py -- truncated N-D Taylor product FP64 GFLOP/s (BASELINE.json's metric) on synthetic dense cubes.

A *step* is one full truncated product Z = X (*) Y of two dense D^n coefficient tensors
(general path, multivariate_taylor.rs:984-1012); default workload = 6 variables x degree 15
(16^6 = 16.8 M coefficients, 128 MiB per tensor, 1.2655e13 algorithmic FLOP), the largest
single-GPU point of BASELINE.json's synthetic sweep.

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload 6x16] [--dump-outputs DIR]

--dump-outputs DIR writes what the timed path computed in its last step, so that two builds can be compared output for
output: DIR/z.npy holds product coefficients (float64) and DIR/z_index.npy their flat positions in Z (float64, exact).
The positions are all of Z when it has at most DUMP_COEFFS coefficients, else a fixed splitmix64 sample, restricted to
the rows the timed path computes (rank 0's rows at N > 1, the CPU sample's rows with --impl reference).  The DFMA
product kernels add partial rows in HBM with RED.ADD.F64, whose order varies, so two runs agree to rounding, not bit
for bit: compare dumps with a relative tolerance (the parity checks below use 1e-12).

N > 1 (launched by torch.distributed.run, one rank per GPU): the SAME product, output rows sharded
over the ranks with the folded-cyclic map of genfer_b200/partition.py; Y lives block-sharded and is
replicated by one NCCL all-gather inside every timed step ("strong" scaling: total work fixed).

Numbers reported (one JSON line, rank 0):
  value     whole-job GFLOP/s, operands resident in HBM, CUDA events, max over ranks
  e2e       same metric through the reference-facing operator (gtp_from_host x2 -> gtp_mul -> gtp_to_host
            at N=1; pinned H2D -> PartitionedProduct -> D2H at N>1) with host buffers
  roofline  product kernel vs the FP64 FMA pipe peak measured live by the library's DFMA probe
  cpu_baseline  the CPU oracle (reference loop order, 1 thread -- the reference is single-threaded)
            on a bounded sample of the same workload, rank 0 at N=1 only
`--impl reference` times that oracle alone (the reference is Rust; no cargo in this image, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "truncated N-D Taylor product FP64 GFLOP/s"
KERNEL_NAMES = {2: "k_mul_blk", 3: "k_mul_slide", 6: "k_mul_blk on zero-extended operands", 7: "k_mul_slide on zero-extended operands"}
UNIT = "GFLOP/s"


def parse_workload(w: str):
    n, d = (int(t) for t in w.lower().split("x"))
    return n, d


def workload_name(n: int, d: int) -> str:
    return f"synthetic TaylorPoly product, {n} vars x degree {d - 1} ({d}^{n} = {d ** n} coefficients per tensor)"


def synth_inputs(n: int, d: int):
    from genfer_b200.synth import SEED_X, SEED_Y, synth_uniform
    shape = (d,) * n
    return synth_uniform(shape, SEED_X), synth_uniform(shape, SEED_Y)


DUMP_COEFFS = 1 << 21   # at most 2 Mi coefficients: values + positions = 32 MiB, a dump small enough to keep beside a run
DUMP_SEED = 20241020


def dump_positions(numel: int) -> np.ndarray:
    """Flat positions in Z written by --dump-outputs: the same for every run and build with the same --workload."""
    if numel <= DUMP_COEFFS:
        return np.arange(numel, dtype=np.int64)
    from genfer_b200.synth import splitmix64
    return np.unique((splitmix64(DUMP_SEED, DUMP_COEFFS) * numel).astype(np.int64))


def write_outputs(out_dir: str, pos: np.ndarray, z: np.ndarray) -> None:
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "z.npy"), np.ascontiguousarray(z, dtype=np.float64))
    np.save(os.path.join(out_dir, "z_index.npy"), pos.astype(np.float64))


# ---------------------------------------------------------------------------------------------
# CPU sample: output rows Z[0, k1, ...] for k1 in `k1s` -- the same loop nest one level down
# (row k0 = 0 of the product only involves X[0], Y[0]), executed by the oracle in reference order.
# ---------------------------------------------------------------------------------------------
def cpu_sample_rows(n: int, d: int, budget_macs: float):
    per_sub = (d * (d + 1) // 2) ** (n - 2)          # MACs of one (n-2)-D sub-product
    k1s, macs = [], 0.0
    for k1 in range(d - 1, -1, -1):                     # heaviest rows first
        if macs + (k1 + 1) * per_sub > budget_macs and k1s:
            break
        k1s.append(k1)
        macs += (k1 + 1) * per_sub
    return sorted(k1s), macs


def run_cpu_sample(x: np.ndarray, y: np.ndarray, k1s):
    """Returns (rows result dict, MACs, seconds).  x, y are the full tensors; only X[0], Y[0] are touched."""
    from oracle import oracle as O
    O.build()
    x0, y0 = np.ascontiguousarray(x[0]), np.ascontiguousarray(y[0])
    t0 = time.perf_counter()
    r, macs = O.mul_rows(x0, y0, x0.shape, k1s)
    dt = time.perf_counter() - t0
    return r, macs, dt


# ---------------------------------------------------------------------------------------------
# Parity samples with k0 > 0: Z[k0, 0..k1, ...] only involves X[:k0+1, :k1+1], Y[:k0+1, :k1+1], and the oracle's
# loop bounds for those output rows are the same on the cut operands as on the full ones (lo = 0, hi = k + 1), so
# the row of the cut product is bit-identical to the oracle's row of the full product.
# ---------------------------------------------------------------------------------------------
def oracle_block(x: np.ndarray, y: np.ndarray, k0: int, k1: int):
    """(Z[k0, 0..k1, ...] by the oracle, MACs)."""
    from oracle import oracle as O
    xc, yc = np.ascontiguousarray(x[:k0 + 1, :k1 + 1]), np.ascontiguousarray(y[:k0 + 1, :k1 + 1])
    r, macs = O.mul_rows(xc, yc, xc.shape, [k0])
    return r[k0], macs


def parity_samples(n: int, d: int, budget_macs: float):
    """(k0, k1) blocks, heaviest leading row first, within the MAC budget."""
    per_sub = float((d * (d + 1) // 2) ** (n - 2))
    picks, macs = [], 0.0
    for k0, k1 in ((d - 1, 0), (d // 2, 1), (1, 3), (d - 2, 1), (3, 2)):
        m = (k0 + 1) * ((k1 + 1) * (k1 + 2) // 2) * per_sub
        if macs + m > budget_macs and picks:
            continue
        picks.append((k0, k1))
        macs += m
    return picks


def run_sweep(ctx, torch, peak_tf: float, cpu_budget_gmac: float):
    """The other points of BASELINE's synthetic sweep (config 4), device-timed like the headline, each with an oracle
    parity sample that includes leading rows k0 > 0."""
    import genfer_b200
    out = []
    # (4,32) .. (5,24): BASELINE's sweep; (4,27), (4,31), (5,17): odd cube edges as evaluation produces them
    # (limit + 1 + sum of orders), zero-extended to the DFMA kernels' extents
    for n, d in ((4, 32), (5, 16), (6, 12), (5, 24), (4, 27), (4, 31), (5, 17)):
        shape = (d,) * n
        xh, yh = synth_inputs(n, d)
        dx, dy = torch.from_numpy(xh).cuda(), torch.from_numpy(yh).cuda()
        dz = torch.empty(shape, dtype=torch.float64, device="cuda")
        rows = list(range(d))
        kind = ctx.mul_kernel_kind(shape, shape, shape)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.mul_rowlist_raw(shape, dx.data_ptr(), shape, dy.data_ptr(), shape, rows, dz.data_ptr())
        torch.cuda.synchronize()
        first_ms = 1e3 * (time.perf_counter() - t0)
        for _ in range(2):
            ctx.mul_rowlist_raw(shape, dx.data_ptr(), shape, dy.data_ptr(), shape, rows, dz.data_ptr())
        reps = 5 if d ** n > 4e6 else 20
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            ctx.mul_rowlist_raw(shape, dx.data_ptr(), shape, dy.data_ptr(), shape, rows, dz.data_ptr())
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        tf = 2.0 * full_macs(n, d) / (ms * 1e-3) / 1e12
        rec = {"workload": f"{n}x{d}", "coefficients": d ** n, "kernel": KERNEL_NAMES.get(kind, "k_mul_ordered"),
               "ms": ms, "tflops": tf, "frac_of_fp64_peak": tf / peak_tf, "first_call_ms": first_ms}
        if cpu_budget_gmac > 0:
            got = dz.cpu().numpy()
            worst, checked, macs = 0.0, 0, 0.0
            for k0, k1 in parity_samples(n, d, cpu_budget_gmac * 1e9):
                ref, m = oracle_block(xh, yh, k0, k1)
                worst = max(worst, float(np.max(np.abs(got[k0, :k1 + 1] - ref) / np.abs(ref))))
                checked += ref.size
                macs += m
            rec["parity"] = {"max_rel_err": worst, "coefficients_checked": checked, "blocks": "Z[k0, 0..k1] incl. k0 > 0",
                             "oracle_macs": macs, "tolerance": 1e-12}
        out.append(rec)
        del dx, dy, dz
    return out


SGCL_DIR = os.path.join(ROOT, "tests", "golden", "sgcl")
# (label, fixture path, --limit override or None, force probabilities on, CPU repetitions)
SGCL_PROGRAMS = [
    ("C1 example --limit 25", "config/example.sgcl", 25, False, 5),
    ("C2 population (= benchmarks/neurips2023/approx/population; 1 var, D~516)", "real_world/population2000.sgcl", None, False, 5),
    ("C2 two_populations (= approx/two_populations; 2 vars, D~336)", "slow/two_populations2000.sgcl", None, False, 2),
    ("C2 population_50_3vars --limit 120, probabilities", "slow/population_50_3vars.sgcl", 120, True, 1),
    ("C2 population_50_4vars --limit 50, probabilities", "slow/population_50_4vars.sgcl", 50, True, 1),
    ("C3 switchpoint", "real_world/switchpoint.sgcl", None, False, 3),
    ("C5 prodigy burglar_alarm", "config/burglar_alarm.sgcl", None, False, 5),
    ("C5 prodigy grass", "config/grass.sgcl", None, False, 5),
]


def run_sgcl_block(ctx, gpu_reps: int = 5):
    """BASELINE metric 2: end-to-end posterior time per .sgcl -- best-of-N wall time through gtp_run_sgcl (source text in,
    report out: the reference's `genfer file.sgcl`), next to the oracle evaluator on one host core, with launches and the
    relative error of Z and p(n)."""
    import genfer_b200
    from oracle import oracle as O
    out = []
    for label, rel, limit, probs_on, cpu_reps in SGCL_PROGRAMS:
        path = os.path.join(SGCL_DIR, rel)
        if not os.path.exists(path):
            alt = [os.path.join(dp, f) for dp, _, fs in os.walk(SGCL_DIR) for f in fs if f == os.path.basename(rel)]
            if not alt:
                out.append({"program": label, "error": "fixture missing"})
                continue
            path = alt[0]
        src = open(path).read()
        opts = genfer_b200.parse_flags(src)
        kw = dict(limit=limit if limit is not None else opts["limit"], no_probs=opts["no_probs"] and not probs_on,
                  no_simplify_gf=opts["no_simplify_gf"], unroll=opts["unroll"])
        tg, launches, g = [], 0, None
        for _ in range(gpu_reps):
            l0 = ctx.launch_count
            t = time.perf_counter()
            g = genfer_b200.run_sgcl(src, ctx=ctx, **kw)
            tg.append(time.perf_counter() - t)
            launches = ctx.launch_count - l0
        to, o = [], None
        for _ in range(cpu_reps):
            t = time.perf_counter()
            o = O.run_sgcl(src, **kw)
            to.append(time.perf_counter() - t)
        zrel = abs(g.total - o.total) / abs(o.total) if o.total else abs(g.total)
        prel = max((abs(a - b) / abs(b) for a, b in zip(g.probs, o.probs) if b), default=0.0)
        out.append({"program": label, "gpu_s": min(tg), "cpu_oracle_s": min(to), "speedup": min(to) / min(tg),
                    "gpu_launches": int(launches), "nodes_evaluated": g.nodes_evaluated, "byte_identical_report": g.report == o.report,
                    "Z_rel_err": zrel, "max_p_rel_err": prel, "gpu_reps": gpu_reps, "cpu_reps": cpu_reps})
    return out


def run_bounds_block(ctx):
    """SURVEY 8 f3: the interval-enclosure run (host evaluator over TaylorPoly<Interval<F64>>, gti_* kernels) -- wall time through
    gtp_run_sgcl_bounds, and for one program the oracle's interval instantiation on one host core beside it."""
    import genfer_b200
    from genfer_b200.interval import run_sgcl_bounds
    from oracle import oracle as O
    out = []
    for label, rel, limit, with_cpu in (("population_50_3vars --limit 60", "slow/population_50_3vars.sgcl", 60, True),
                                        ("two_populations2000", "slow/two_populations2000.sgcl", None, False)):
        path = os.path.join(SGCL_DIR, rel)
        if not os.path.exists(path):
            out.append({"program": label, "error": "fixture missing"})
            continue
        src = open(path).read()
        opts = genfer_b200.parse_flags(src)
        g = genfer_b200.run_sgcl(src, limit=limit if limit is not None else opts["limit"], no_simplify_gf=opts["no_simplify_gf"],
                                 unroll=opts["unroll"], ctx=ctx)
        n, tg, launches, b = len(g.probs), [], 0, None
        for _ in range(3):
            l0 = ctx.launch_count
            t = time.perf_counter()
            b = run_sgcl_bounds(src, limit=n, unroll=opts["unroll"], ctx=ctx)
            tg.append(time.perf_counter() - t)
            launches = ctx.launch_count - l0
        inside = b.total[0] <= g.total <= b.total[1] and all(lo <= p <= hi for p, (lo, hi) in zip(g.probs, b.probs))
        rec = {"program": label, "gpu_bounds_s": min(tg), "gpu_launches": int(launches), "f64_results_inside": bool(inside),
               "Z_enclosure": list(b.total)}
        if with_cpu:
            t = time.perf_counter()
            o = O.run_sgcl_bounds(src, limit=n, unroll=opts["unroll"])
            rec["cpu_oracle_bounds_s"] = time.perf_counter() - t
            rec["speedup"] = rec["cpu_oracle_bounds_s"] / rec["gpu_bounds_s"]
            rec["overlaps_oracle"] = bool(max(b.total[0], o.total[0]) <= min(b.total[1], o.total[1]))
        out.append(rec)
    return out


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, ln in self.lines:
            f = [c.strip() for c in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            smax = mx
            if t0 <= t <= t1 + 0.1:
                sm.append(clk)
                try:
                    power.append(float(f[3]))
                except ValueError:
                    pass
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        if not sm:  # region shorter than one sample: take the nearest ones
            sm = [float(ln.split(",")[1]) for _, ln in self.lines[-3:] if len(ln.split(",")) >= 9] or [0.0]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path.  The reference is Rust and cannot be built in this
    image (no cargo/rustc), so this is the oracle port: same loop order, separate multiply and add, 1 thread
    (the reference is single-threaded: src/main.rs:96-106, every IR node is an Rc)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, d = parse_workload(args.workload)
    x, y = synth_inputs(n, d)
    k1s, _ = cpu_sample_rows(n, d, budget_macs=args.cpu_budget_gmac * 1e9 * 0.4)
    times, macs = [], 0.0
    for i in range(args.warmup + args.steps):
        r, macs, dt = run_cpu_sample(x, y, k1s)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:   # r holds rows k1s of X[0] (*) Y[0], i.e. Z[0, k1, ...]: the positions below d^(n-1)
        pos = dump_positions(d ** n)
        pos = pos[(pos < d ** (n - 1)) & np.isin(pos // d ** (n - 2), k1s)]
        write_outputs(args.dump_outputs, pos, r.reshape(-1)[pos])
    total = sum(times)
    value = 2.0 * macs * len(times) / total / 1e9
    sample = (f"output rows Z[0, k1, ...], k1 in {k1s[0]}..{k1s[-1]} of the {workload_name(n, d)}: "
              f"{macs:.4g} MACs per step (of {full_macs(n, d):.4g}), oracle port in reference loop order, "
              f"g++ -O3 -march=native -ffp-contract=off")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(n, d), "inputs": "iid uniform [0,1), splitmix64 seeds 20230517/20231210"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                             "host_cores": host_cores()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def full_macs(n: int, d: int) -> float:
    return float((d * (d + 1) // 2) ** n)


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import genfer_b200
    from genfer_b200.partition import PartitionedProduct, gpu_row_kernel, rows_for_rank, shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the f64 Taylor path has no CPU fallback "
                         "(use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n, d = parse_workload(args.workload)
    shape = (d,) * n
    K, W = args.steps, args.warmup
    flops = 2.0 * full_macs(n, d)

    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    if world > 1:
        # group context: the partitioning, the NCCL all-gather and the row-sharded result live INSIDE the library, behind
        # the same gtp_mul a single-GPU caller uses (torch.distributed only ships the 128-byte NCCL id)
        ids = [genfer_b200.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx = genfer_b200.Context.create_group(local, rank, world, ids[0], stream=stream.cuda_stream)
        if d ** n < 10 ** 7:   # gtp_mul partitions from 1e7 result coefficients by default (north_star); smaller sweep points on request
            ctx.set_partition_threshold(d ** n)
    else:
        ctx = genfer_b200.Context(local, stream=stream.cuda_stream)
    kind = ctx.mul_kernel_kind(shape, shape, shape)

    xh_np, yh_np = synth_inputs(n, d)
    hx = torch.from_numpy(xh_np).pin_memory()
    hy = torch.from_numpy(yh_np).pin_memory()
    dx = hx.to("cuda", non_blocking=True)
    dy = hy.to("cuda", non_blocking=True)
    pp = PartitionedProduct(shape, shape, shape, gpu_row_kernel(ctx))
    y_shard = pp.shard_of(dy) if world > 1 else dy
    lo, hi, block = shard_bounds(d, world, rank)
    hy_shard = torch.zeros((block,) + shape[1:], dtype=torch.float64).pin_memory()
    hy_shard[: hi - lo] = hy[lo:hi]
    hx_shard = torch.zeros((block,) + shape[1:], dtype=torch.float64).pin_memory()
    hx_shard[: hi - lo] = hx[lo:hi]
    TXd = genfer_b200.TaylorPoly.from_device(dx.data_ptr(), shape, shape, ctx)   # X resident and replicated
    out_rows = torch.empty((len(pp.rows),) + shape[1:], dtype=torch.float64, device="cuda")
    h_out = torch.empty((len(pp.rows),) + shape[1:], dtype=torch.float64).pin_memory()
    row_kernel = gpu_row_kernel(ctx)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()

    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]

    def step(i=None):
        if world == 1:
            if i is not None:
                kev[i][0].record()
            row_kernel(shape, dx, shape, dy, shape, pp.rows, out_rows)
            if i is not None:
                kev[i][1].record()
            return None
        # N > 1: Y lives block-sharded; gtp_mul replicates it (ncclAllGather over NVLink, inside the library), computes
        # this rank's folded-cyclic rows and leaves the result row-sharded
        TY = genfer_b200.TaylorPoly.from_device_block(y_shard.data_ptr(), shape, shape, ctx)
        TY.replicate()
        if i is not None:
            kev[i][0].record()
        Z = TXd * TY
        if i is not None:
            kev[i][1].record()
        return Z

    # ---- device-resident timing ------------------------------------------------------------
    torch.cuda.synchronize()
    t_first0 = time.perf_counter()
    step()                                # first call: builds and uploads the kernel's step / unit tables (plan cache miss)
    torch.cuda.synchronize()
    first_call_ms = 1e3 * (time.perf_counter() - t_first0)
    for _ in range(max(W - 1, 0)):
        step()
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    torch.cuda.synchronize()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    for i in range(K - 1):
        step(i)
    z_last = step(K - 1)                  # the product at N > 1 (None at N = 1: it is in out_rows)
    e1.record()
    torch.cuda.synchronize()
    barrier()
    t_host1 = time.perf_counter()
    launches = ctx.launch_count - l0
    clocks = sampler.stop(t_host0, t_host1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        rows = pp.rows if world == 1 else z_last.local_rows()   # the rows of Z this rank holds, in the order it holds them
        row_len = d ** (n - 1)
        slot = np.full(d, -1, dtype=np.int64)
        slot[rows] = np.arange(len(rows))
        pos = dump_positions(d ** n)
        pos = pos[slot[pos // row_len] >= 0]
        at = slot[pos // row_len] * row_len + pos % row_len
        if world == 1:
            z = out_rows.view(-1)[torch.from_numpy(at).cuda()].cpu().numpy()
        else:
            held = np.empty(len(rows) * row_len)
            z_last.to_host_local_ptr(held.ctypes.data)
            z = held[at]
        write_outputs(args.dump_outputs, pos, z)
    del z_last
    ms_total = e0.elapsed_time(e1)
    ms_kernel = sum(a.elapsed_time(b) for a, b in kev) / K
    t = torch.tensor([ms_total, ms_kernel], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_kernel_max = float(t[0]), float(t[1])
    value = flops * K / (ms_total * 1e-3) / 1e9

    # ---- end to end with host buffers ----------------------------------------------------------
    def e2e_step():
        if world == 1:   # the reference-facing operator surface through the C ABI
            X = genfer_b200.TaylorPoly.from_host_ptr(hx.data_ptr(), shape, shape, ctx)
            Y = genfer_b200.TaylorPoly.from_host_ptr(hy.data_ptr(), shape, shape, ctx)
            Z = X * Y
            Z.to_host_ptr(h_out.data_ptr())               # synchronises
        else:             # the same operator surface on a group context: block-sharded uploads (1/N of the H2D traffic
            X = genfer_b200.TaylorPoly.from_host_block_ptr(hx_shard.data_ptr(), shape, shape, ctx)   # per rank), NVLink
            Y = genfer_b200.TaylorPoly.from_host_block_ptr(hy_shard.data_ptr(), shape, shape, ctx)   # all-gathers,
            Z = X * Y                                                                                   # partitioned product,
            Z.to_host_local_ptr(h_out.data_ptr())                                                       # D2H of this rank's rows

    for _ in range(min(W, 2)):
        e2e_step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    te = torch.tensor([t1 - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = flops * K / float(te[0]) / 1e9
    h2d = (hx.numel() + hy.numel()) * 8 if world == 1 else (hx_shard.numel() + hy_shard.numel()) * 8
    d2h = h_out.numel() * 8
    e2e_out_sample = h_out[0, :].clone() if rank == 0 else None   # Z[0, ...] (row 0 belongs to rank 0)

    # ---- roofline of the product kernel ---------------------------------------------------------
    my_rows_macs = sum(k + 1 for k in pp.rows) * float((d * (d + 1) // 2) ** (n - 1))
    achieved = 2.0 * my_rows_macs / (ms_kernel * 1e-3) / 1e12           # this rank's launch
    peak_fl, _ = ctx.fp64_peak_probe(0, 16384)
    peak = peak_fl / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "product_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.workload, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "fp64", "kernel": KERNEL_NAMES.get(kind, "k_mul_ordered"),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": traffic,
                "peak_source": "FP64 FMA pipe measured live by gtp_fp64_peak_probe (8 independent DFMA chains/thread, all SMs); "
                               "MEASURED_PEAKS.json has no FP64 entry; DMMA m8n8k4 measures the same rate (profiles/fp64_peaks.json)",
                "algorithmic_flop_per_launch": 2.0 * my_rows_macs, "kernel_ms": ms_kernel}

    # ---- HBM-bound axis reduction on the same tensors (Metric 1b, shift_down) ---------------------
    aux = []
    if world == 1 and not args.no_aux:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
        hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if os.path.exists(peaks_path) else "6.65 TB/s (of fallback)"
        TX = genfer_b200.TaylorPoly.from_device(dx.data_ptr(), shape, shape, ctx)
        TY = genfer_b200.TaylorPoly.from_device(dy.data_ptr(), shape, shape, ctx)
        for v, nm in ((n - 1, "last axis"), (0, "first axis")):
            for _ in range(3):
                TX.shift_down(v, d - 1), TY.shift_down(v, d - 1)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            a.record()
            for i in range(reps):                           # alternate X / Y (each 128 MiB > L2) so reads come from HBM
                (TX if i % 2 == 0 else TY).shift_down(v, d - 1)
            b.record()
            torch.cuda.synchronize()
            msr = a.elapsed_time(b) / reps
            nbytes = 8.0 * (d ** n + d ** (n - 1))
            aux.append({"kernel": f"shift_down({nm}, n={d - 1}): full axis reduction", "bound": "hbm",
                        "achieved": nbytes / (msr * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": nbytes / (msr * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": nbytes,
                        "ms": msr, "peak_source": hbm_src})

    # ---- CPU baseline + parity on the sample (rank 0, N = 1) ---------------------------------------
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        k1s, _ = cpu_sample_rows(n, d, budget_macs=args.cpu_budget_gmac * 1e9)
        r, macs, dt = run_cpu_sample(xh_np, yh_np, k1s)
        cpu = {"value": 2.0 * macs / dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"output rows Z[0, k1, ...], k1 in {k1s[0]}..{k1s[-1]} of the same product: {macs:.4g} MACs "
                         f"in {dt:.1f} s; oracle port, reference loop order, 1 thread (the reference is single-threaded)",
               "host_cores": host_cores(), "seconds": dt}
        got = e2e_out_sample.numpy()[k1s]
        ref = r[k1s]
        parity = {"vs": "oracle, same inputs, rows Z[0, k1, ...] of the e2e result",
                  "max_rel_err": float(np.max(np.abs(got - ref) / np.abs(ref))), "tolerance": 1e-12,
                  "coefficients_checked": int(ref.size)}
        # leading rows k0 > 0 (every j0 <= k0 slab pair contributes): blocks Z[k0, 0..k1, ...]
        full = h_out.numpy()
        worst, checked, bmacs = 0.0, 0, 0.0
        for k0, k1 in parity_samples(n, d, args.cpu_budget_gmac * 1e9 * 0.5):
            bref, m = oracle_block(xh_np, yh_np, k0, k1)
            worst = max(worst, float(np.max(np.abs(full[k0, :k1 + 1] - bref) / np.abs(bref))))
            checked += bref.size
            bmacs += m
        parity["k0_gt_0"] = {"blocks": "Z[k0, 0..k1, ...] for (k0, k1) in " + str(parity_samples(n, d, args.cpu_budget_gmac * 1e9 * 0.5)),
                             "max_rel_err": worst, "coefficients_checked": int(checked), "oracle_macs": bmacs}
        parity["max_rel_err"] = max(parity["max_rel_err"], worst)
        parity["coefficients_checked"] += int(checked)

    if rank == 0 and world > 1 and not args.no_cpu:
        # N > 1: a small oracle sample of rank 0's own rows of the partitioned e2e result (no CPU baseline here: that is N = 1's)
        budget = min(args.cpu_budget_gmac, 4.0) * 1e9
        k1s, _ = cpu_sample_rows(n, d, budget_macs=budget)
        r, macs, dt = run_cpu_sample(xh_np, yh_np, k1s)
        got, ref = e2e_out_sample.numpy()[k1s], r[k1s]
        parity = {"vs": "oracle, same inputs, rows Z[0, k1, ...] and blocks Z[k0 > 0, 0..k1, ...] of rank 0's share of the partitioned e2e result",
                  "max_rel_err": float(np.max(np.abs(got - ref) / np.abs(ref))), "tolerance": 1e-12,
                  "coefficients_checked": int(ref.size), "oracle_seconds": dt}
        local = h_out.numpy()
        mine = {int(k0): i for i, k0 in enumerate(pp.rows)}
        blocks = [(k0, k1) for k0, k1 in parity_samples(n, d, budget) if k0 in mine]
        for k0, k1 in blocks:
            bref, _ = oracle_block(xh_np, yh_np, k0, k1)
            parity["max_rel_err"] = max(parity["max_rel_err"], float(np.max(np.abs(local[mine[k0], :k1 + 1] - bref) / np.abs(bref))))
            parity["coefficients_checked"] += int(bref.size)
        parity["k0_gt_0_blocks"] = str(blocks)

    sweep, sgcl, bounds = None, None, None
    if rank == 0 and world == 1 and not args.no_sweep:
        sweep = run_sweep(ctx, torch, peak, 0.0 if args.no_cpu else args.cpu_budget_gmac * 0.1)
    if rank == 0 and world == 1 and not args.no_sgcl:
        sgcl = run_sgcl_block(ctx)
        bounds = run_bounds_block(ctx)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(n, d),
                           "inputs": "iid uniform [0,1), splitmix64 seeds 20230517/20231210; X, Y, Z = "
                                     f"{3 * d ** n * 8 / 2 ** 20:.0f} MiB" + (" > 126 MB L2 (inputs larger than L2)" if 3 * d ** n * 8 > 126e6 else
                                                                               " (fits L2; compute-bound kernel, arithmetic intensity > 1 kFLOP/B)"),
                           "parallelism": "1 GPU" if world == 1 else
                           f"output rows folded-cyclic over {world} GPUs inside gtp_mul (group context), Y block-sharded + in-library NCCL all-gather per step",
                           "kernel": roofline["kernel"]},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "api": "gtp_from_host x2 -> gtp_mul -> gtp_to_host" if world == 1 else
                               "gtp_from_host_block x2 (X, Y block shards) -> gtp_mul on a group context (in-library ncclAllGather x2, "
                               "partitioned rows) -> gtp_to_host_local (this rank's rows)"},
                "gpu_launches": int(launches),
                "roofline": roofline, "aux_rooflines": aux, "cpu_baseline": cpu, "parity": parity,
                "kernel_ms_max_over_ranks": ms_kernel_max,
                "first_call": {"ms": first_call_ms, "steady_ms": ms_total / K,
                               "note": "first product of a shape builds + uploads the kernel's step/unit tables (host) and synchronises once"},
                "sweep": sweep, "sgcl": sgcl, "bounds": bounds}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="6x16", help="NxD: N variables, cube edge D (degree D-1)")
    ap.add_argument("--cpu-budget-gmac", type=float, default=40.0, help="size of the CPU sample in GMAC")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the other four points of the synthetic sweep")
    ap.add_argument("--no-sgcl", action="store_true", help="skip the end-to-end .sgcl block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's product (sampled) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
