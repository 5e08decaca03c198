"""Fixed-iteration timing of the tiled engine at k = 32, 48 and 64: the tensor-core passes (engine=2: tcgen05 for Float32,
DMMA for Float64) against the scalar-FMA pass (engine=4) on the same shapes, in one process.

    python tools/large_k_bench.py [--iters N] [--out FILE]

Shapes: C3 (10000 x 10000 Float32, 64 restarts) and C4 (100000 x 2000 Float64, 32 restarts).  Algorithmic rate = 8nmk flops per
restart-iteration (as bench.py) over the host time of the solve (which ends in a device synchronisation), next to the
share of measure_peak(13) / 3 (tcgen05 kind::tf32 with the 3-term split: three MMAs per product) for Float32 and of
measure_peak(1) (FP64 DMMA) for Float64.  The card name and power limit are read in the same process.  JSON lines on stdout
(and appended to --out).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nmfk.jl_b200", "python"))
import numpy as np  # noqa: E402
import nmfk_b200 as nb  # noqa: E402
from nmfk_b200 import synth  # noqa: E402

SHAPES = [("C3", 10000, 10000, np.float32, 64), ("C4", 100000, 2000, np.float64, 32)]
KS = (32, 48, 64)


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    with nb.Context(0) as ctx:
        peaks = dict(tf32_3term=max(ctx.measure_peak(13) for _ in range(2)) / 3, dmma=max(ctx.measure_peak(1) for _ in range(2)))
        emit(dict(card=card(), peaks_tflops=peaks))
        for name, n, m, dt, R in SHAPES:
            X = synth.mixture(n, m, 16, seed=2015, dtype=dt)
            ctx.set_X(X)
            del X
            peak = peaks["tf32_3term"] if dt == np.float32 else peaks["dmma"]
            for k in KS:
                for engine in (2, 4):
                    ms = None
                    for iters in (10, args.iters, args.iters):  # warm-up (one objective check loads every kernel), best of two
                        b = ctx.batch(k, R)
                        b.init_random(2015)
                        ctx.solve([b], nb.default_params(maxiter=iters, engine=engine, normalize=0))
                        out = b.get(factors=False)
                        b.close()
                        if iters == args.iters and (ms is None or ctx.last_solve_ms < ms):
                            ms = ctx.last_solve_ms
                    tot = int(out["iters"].sum())
                    flops = 8.0 * n * m * k * tot
                    emit(dict(shape=name, n=n, m=m, k=k, R=R, dtype=np.dtype(dt).name, engine=engine, restart_iters=tot,
                              ms=round(ms, 2), rit_per_s=round(tot / ms * 1e3, 2), tflops=round(flops / ms / 1e9, 2),
                              share_of_peak=round(flops / ms / 1e9 / peak, 4)))


if __name__ == "__main__":
    main()
