#!/usr/bin/env python3
"""Generates tests/golden/tc2_pass.npz: a compact record of the factors, iteration counts, stop reasons and objectives of small
Float32 solves that run the second-generation tcgen05 pass (k <= 16, kl_tiled_tc2.cu) on a B200.  Output of the pass is meant
to stay bit-identical across rewrites of its schedule, so tests/test_gpu_tc2_images.py compares a fresh run with this record by
np.array_equal.

Record of one output array (see `compact`): arrays of at most 64 entries are kept whole; a larger one (W, H) is kept as the
SHA-256 digest of its bytes (any changed bit changes it) plus its entries at 64 fixed positions, which say by how much a
mismatching run differs.  The file stays a few kilobytes instead of megabytes of incompressible Float32 factors.

The committed file was written by this script from the tc2 pass as it stood before V operand images were built by a producer
kernel (the pass then staged them itself with four warps and read X own-contiguous).

    python tests/golden/make_tc2_golden.py [OUT.npz]      # needs the built package and a GPU

The cases cover k = 1, 5, 8, 9, 12, 16; own / step sizes that are not multiples of 128 / 64; odd restart counts (shadow units);
restarts that stop at different iterations while others keep running; sliced reductions (S > 1) and single-slice launches;
normalizevector, Hfixed and Wfixed.
"""
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "nmfk.jl_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "tc2_pass.npz")

# name, n, m, k, R, solver keywords, normalizevector
CASES = [
    ("k1_r3", 260, 132, 1, 3, dict(maxiter=5), False),
    ("k5_r5_stops", 1000, 332, 5, 5, dict(maxiter=60, tol=5000.0), False),
    ("k8_r4_sliced", 3108, 200, 8, 4, dict(maxiter=4), False),
    ("k9_r7_normvec", 1156, 840, 9, 7, dict(maxiter=6), True),
    ("k16_r5", 1028, 516, 16, 5, dict(maxiter=4, normalize=0), False),
    ("k16_r2_hfixed", 644, 388, 16, 2, dict(maxiter=5, Hfixed=1), False),
    ("k12_r3_wfixed", 388, 1284, 12, 3, dict(maxiter=5, Wfixed=1), False),
]

NSAMPLE = 64


def compact(res):
    """name -> array  ==>  the record compared by the test (same keys for small arrays; key + '_sha256' / '_sample' otherwise)."""
    out = {}
    for key, val in res.items():
        val = np.ascontiguousarray(val)
        if val.size <= NSAMPLE:
            out[key] = val
            continue
        out[key + "_sha256"] = np.frombuffer(hashlib.sha256(val.tobytes()).digest(), dtype=np.uint8)
        pos = np.random.default_rng(val.size).choice(val.size, NSAMPLE, replace=False)
        out[key + "_sample"] = val.reshape(-1)[np.sort(pos)]
    return out


def run_case(ctx, case):
    import nmfk_b200 as nb
    from nmfk_b200 import synth

    name, n, m, k, R, kw, normvec = case
    X = synth.mixture(n, m, min(k, 4), seed=n + m + k, dtype=np.float32)
    W0, H0 = synth.philox_inits(1000 + k, R, n, k, m, dtype=np.float32)
    nv = (1.0 + np.arange(n, dtype=np.float32) % 7) if normvec else None
    ctx.set_X(X, normalizevector=nv)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(engine=2, **kw))
    g = b.get()
    b.close()
    return {name + "_" + key: np.asarray(g[key]) for key in ("W", "H", "iters", "stop_reason", "obj_ssq")}


if __name__ == "__main__":
    import nmfk_b200 as nb

    out = {}
    with nb.Context(0) as ctx:
        for case in CASES:
            res = run_case(ctx, case)
            out.update(compact(res))
            print(case[0], "iters", res[case[0] + "_iters"].tolist(), "stop", res[case[0] + "_stop_reason"].tolist())
    np.savez_compressed(sys.argv[1] if len(sys.argv) > 1 else GOLDEN, **out)
