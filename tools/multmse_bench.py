"""Restart-iterations/s of Variant KL_DIV (method=:nmf, algorithm=:multmse) against method=:simple on the same shapes, in one
process, the two variants alternating (simple, multmse, simple, multmse, ...) so that clock and neighbour drift hits both.

    python tools/multmse_bench.py [--iters N] [--reps N] [--out FILE] [--timing]

Cases: the C3 matrix (10000 x 10000 Float32) at k = 16 (tc2_pass_kernel) and k = 24 (tc_pass_kernel), 64 restarts, and the C4
matrix (100000 x 2000 Float64) at k = 32 (tiled_dmma_pass_kernel), 32 restarts; fixed iteration counts (tol = 0, so neither
variant stops early).  Time = device time of the solve (CUDA events around it, nmfk_last_solve_ms), best of --reps, after one
warm-up solve of each variant.  The card name and power limit are read in the same process.  JSON lines on stdout (and appended
to --out).  --timing: one more solve of each variant per case with NMFK_TILED_TIMING=1, whose per-phase line goes to stderr.
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

CASES = [("C3", 10000, 10000, np.float32, 16, 64), ("C3_k24", 10000, 10000, np.float32, 24, 64),
         ("C4_k32", 100000, 2000, np.float64, 32, 32)]
VARIANTS = (("simple", 0), ("multmse", 3))


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--timing", action="store_true")
    args = ap.parse_args()

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    def solve(ctx, k, R, variant, iters):
        b = ctx.batch(k, R)
        b.init_random(2015)
        ctx.solve([b], nb.default_params(variant=variant, maxiter=iters, tol=0.0, normalize=0))
        tot = int(b.get(factors=False)["iters"].sum())
        b.close()
        return tot, ctx.last_solve_ms

    with nb.Context(0) as ctx:
        emit(dict(card=card()))
        for name, n, m, dt, k, R in CASES:
            X = synth.mixture(n, m, 16, seed=2015, dtype=dt)
            ctx.set_X(X)
            del X
            for _, v in VARIANTS:  # warm-up: module loads, pool growth
                solve(ctx, k, R, v, 10)
            best = {}
            for _ in range(args.reps):
                for vname, v in VARIANTS:
                    tot, ms = solve(ctx, k, R, v, args.iters)
                    if vname not in best or ms < best[vname][1]:
                        best[vname] = (tot, ms)
            rate = {vname: tot / ms * 1e3 for vname, (tot, ms) in best.items()}
            for vname, (tot, ms) in best.items():
                emit(dict(case=name, n=n, m=m, k=k, R=R, dtype=np.dtype(dt).name, variant=vname, restart_iters=tot, ms=round(ms, 2),
                          rit_per_s=round(rate[vname], 2)))
            emit(dict(case=name, multmse_over_simple_time_per_iteration=round(rate["simple"] / rate["multmse"], 4)))
            if args.timing:
                os.environ["NMFK_TILED_TIMING"] = "1"
                for vname, v in VARIANTS:
                    print("[%s %s]" % (name, vname), file=sys.stderr, flush=True)
                    solve(ctx, k, R, v, args.iters)
                del os.environ["NMFK_TILED_TIMING"]


if __name__ == "__main__":
    main()
