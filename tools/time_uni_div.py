"""Per-op `gtu_div` (k_uni_div) time of one built libgenfer_taylor.so, so that two builds can be compared in one session.

Runs on a torch stream that the context adopts and times `--calls` back-to-back quotients of seeded Polynomials per order with CUDA
events (one kernel each, plus the stream-ordered allocation of the result).  Also prints a hash of the result bits, which
must agree between builds.  One JSON line per order.
usage: time_uni_div.py --lib path/to/libgenfer_taylor.so [--label NAME] [--calls N]"""
import argparse
import ctypes as C
import hashlib
import json

import numpy as np
import torch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", required=True)
    ap.add_argument("--label", default="")
    ap.add_argument("--calls", type=int, default=200)
    a = ap.parse_args()
    lib = C.CDLL(a.lib)
    vp, f64p = C.c_void_p, C.POINTER(C.c_double)
    lib.gtp_ctx_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    lib.gtp_ctx_destroy.argtypes = [vp]
    lib.gtu_from_coefficients.argtypes = [vp, f64p, C.c_uint64, C.POINTER(vp)]
    lib.gtu_div.argtypes = [vp, vp, vp, C.POINTER(vp)]
    lib.gtu_free.argtypes = [vp, vp]
    lib.gtu_to_host.argtypes = [vp, vp, f64p]
    torch.cuda.init()
    stream = torch.cuda.Stream()   # a stream of its own: the default stream's handle is 0, which the library reads as "none"
    ctx = vp()
    assert lib.gtp_ctx_create(0, vp(stream.cuda_stream), C.byref(ctx)) == 0
    name = torch.cuda.get_device_name(0)
    for n in (64, 257, 1000, 2048):
        rng = np.random.default_rng(n)
        xs = [np.ascontiguousarray(rng.uniform(-1, 1, n) * 0.9 ** np.arange(n)) for _ in range(2)]
        xs[1][0] = 1.25
        h = [vp(), vp()]
        for x, hh in zip(xs, h):
            assert lib.gtu_from_coefficients(ctx, x.ctypes.data_as(f64p), n, C.byref(hh)) == 0

        def div():
            o = vp()
            assert lib.gtu_div(ctx, h[0], h[1], C.byref(o)) == 0
            return o

        o = div()   # warm-up, and the bits to hash
        out = np.empty(n)
        assert lib.gtu_to_host(ctx, o, out.ctypes.data_as(f64p)) == 0
        lib.gtu_free(ctx, o)
        best = None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            outs = []
            e0.record(stream)
            for _ in range(a.calls):
                outs.append(div())
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / a.calls
            best = ms if best is None else min(best, ms)
            for x in outs:
                lib.gtu_free(ctx, x)
        for hh in h:
            lib.gtu_free(ctx, hh)
        print(json.dumps({"label": a.label, "gpu": name, "order": n, "us_per_div": round(best * 1e3, 2),
                          "bits_sha1": hashlib.sha1(out.tobytes()).hexdigest()[:16]}), flush=True)
    lib.gtp_ctx_destroy(ctx)


if __name__ == "__main__":
    main()
