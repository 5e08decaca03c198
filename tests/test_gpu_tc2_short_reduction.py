"""The second-generation tcgen05 pass (k <= 16, kl_tiled_tc2.cu) on reductions shorter than its three X tile stages: one or two
64-step chunks per half-update, so the load warp issues every X tile up front and never waits for a stage to be released.  One
restart per CTA group (a shadow unit) against the Float64 oracle, iteration by iteration, and batches of several restarts (whole
and odd groups) against the scalar-FMA pass of the tiled engine, with the tolerances of test_gpu_parity.py."""
import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu

RTOL32 = 1e-4


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


# (n, m): the W-update reduces over m, the H-update over n
@pytest.mark.parametrize("n,m,k,niter", [(1000, 100, 9, 12), (64, 1204, 16, 10), (128, 124, 5, 15)])
def test_short_reduction_trace_matches_oracle(ctx, n, m, k, niter):
    X = synth.mixture(n, m, 3, seed=n + m, dtype=np.float32)
    W0, H0 = synth.philox_inits(7 + k, 1, n, k, m, dtype=np.float32)
    Wt, Ht, _ = nb.trace(X, k, W0[0], H0[0], niter, ctx=ctx, engine=2)
    Ws, Hs = [], []
    o.nmf_multiplicative(np.array(X, dtype=np.float64, order="F"), k, Winit=W0[0].astype(np.float64), Hinit=H0[0].astype(np.float64),
                         maxiter=niter, trace=lambda it, W, H, obj: (Ws.append(W.copy()), Hs.append(H.copy())))
    for t in range(niter):
        assert relerr(Wt[t], Ws[t]) < RTOL32, ("W", t)
        assert relerr(Ht[t], Hs[t]) < RTOL32, ("H", t)


@pytest.mark.parametrize("n,m,k,R", [(1028, 40, 5, 7), (120, 2000, 12, 4), (260, 128, 16, 9)])
def test_short_reduction_batches_match_scalar_pass(ctx, n, m, k, R):
    X = synth.mixture(n, m, min(k, 4), seed=3 * n + m, dtype=np.float32)
    W0, H0 = synth.philox_inits(50 + R, R, n, k, m, dtype=np.float32)
    ctx.set_X(X)
    out = []
    for eng in (2, 4):
        b = ctx.batch(k, R)
        b.set_init(W0, H0)
        ctx.solve([b], nb.default_params(maxiter=4, engine=eng))
        g = b.get()
        out.append((g["W"], g["H"]))
        b.close()
    assert relerr(out[0][0], out[1][0]) < 2e-5 and relerr(out[0][1], out[1][1]) < 2e-5
