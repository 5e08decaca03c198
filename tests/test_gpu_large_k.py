"""k from 33 to 64 on the tiled engine (the resident engines stop at 32): the scalar-FMA pass, the Float64 DMMA pass and the
Float32 tcgen05 pass (one restart per CTA at k > 32) against the CPU oracle, through every entry point that reaches the
tiled engine.  Tolerances as in test_gpu_parity.py."""
import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu

RTOL64 = 1e-9
RTOL32 = 1e-4


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def oracle_trace(X, k, W0, H0, niter, **kw):
    Ws, Hs = [], []

    def cb(it, W, H, obj):
        Ws.append(W.copy())
        Hs.append(H.copy())

    Xc = np.array(X, dtype=np.float64, order="F", copy=True)
    o.nmf_multiplicative(Xc, k, Winit=W0.astype(np.float64), Hinit=H0.astype(np.float64), maxiter=niter, trace=cb, **kw)
    return np.stack(Ws), np.stack(Hs)


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


# engine=2: DMMA pass (Float64) / tcgen05 pass (Float32, row and column counts multiples of 4); engine=4: scalar-FMA pass
@pytest.mark.parametrize("n,m,k,dt,engine", [(701, 299, 33, np.float64, 2), (520, 390, 40, np.float64, 2),
                                             (333, 1025, 48, np.float64, 2), (611, 203, 53, np.float64, 2),
                                             (900, 260, 64, np.float64, 2),
                                             (701, 299, 33, np.float64, 4), (520, 390, 40, np.float64, 4),
                                             (333, 1025, 48, np.float64, 4), (611, 203, 53, np.float64, 4),
                                             (900, 260, 64, np.float64, 4),
                                             (700, 300, 33, np.float32, 2), (520, 388, 40, np.float32, 2),
                                             (332, 1024, 48, np.float32, 2), (900, 260, 64, np.float32, 2)])
def test_large_k_trace_parity(ctx, n, m, k, dt, engine):
    niter = 10
    X = synth.mixture(n, m, 5, seed=17, dtype=dt)
    W0, H0 = synth.philox_inits(23, 1, n, k, m, dtype=dt)
    Wt, Ht, ob = nb.trace(X, k, W0[0], H0[0], niter, ctx=ctx, engine=engine)
    Wr, Hr = oracle_trace(X, k, W0[0], H0[0], niter)
    tol = RTOL64 if dt == np.float64 else RTOL32
    for t in range(niter):
        assert relerr(Wt[t], Wr[t]) < tol, ("W", t)
        assert relerr(Ht[t], Hr[t]) < tol, ("H", t)


def test_large_k_tc_random_shapes_match_scalar_pass(ctx):
    """Ragged shapes through the tcgen05 pass and the scalar-FMA pass: own / reduction sizes that are not multiples of the
    128 x 64 tile, sliced reductions, 1..5 restarts, k = 33..64."""
    rng = np.random.default_rng(321)
    for c in range(8):
        n = int(rng.choice([4, 132, 260, 1000, 3108])) if c % 3 else 4 * int(rng.integers(1, 500))
        m = 4 * int(rng.integers(1, 400)) if c % 2 else int(rng.choice([4, 68, 332, 2000]))
        k, R, iters = int(rng.integers(33, 65)), int(rng.integers(1, 6)), int(rng.integers(1, 5))
        X = synth.mixture(n, m, 4, seed=c, dtype=np.float32)
        W0, H0 = synth.philox_inits(100 + c, R, n, k, m, dtype=np.float32)
        ctx.set_X(X)
        out = []
        for eng in (2, 4):
            b = ctx.batch(k, R)
            b.set_init(W0, H0)
            ctx.solve([b], nb.default_params(maxiter=iters, engine=eng))
            g = b.get()
            out.append((g["W"], g["H"], g["obj_norm"]))
            b.close()
        assert relerr(out[0][0], out[1][0]) < 2e-5 and relerr(out[0][1], out[1][1]) < 2e-5, (c, n, m, k, R, iters)
        assert np.allclose(out[0][2], out[1][2], rtol=1e-4), (c, n, m, k, R, iters)


@pytest.mark.parametrize("k,dt", [(40, np.float32), (56, np.float32), (64, np.float32), (40, np.float64), (56, np.float64),
                                  (64, np.float64)])
def test_large_k_engine2_runs_the_tensor_pass(ctx, k, dt):
    """engine=2 and engine=4 agree to rounding but not bit for bit: the tensor-core pass (tcgen05 / DMMA), not the scalar-FMA
    pass, ran under engine=2."""
    n, m, R = 520, 388, 2
    X = synth.mixture(n, m, 4, seed=3, dtype=dt)
    W0, H0 = synth.philox_inits(8, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    out = {}
    for eng in (2, 4):
        b = ctx.batch(k, R)
        b.set_init(W0, H0)
        ctx.solve([b], nb.default_params(maxiter=6, engine=eng, normalize=0))
        out[eng] = b.get()
        b.close()
    tol = 1e-10 if dt == np.float64 else 2e-5
    assert relerr(out[2]["W"], out[4]["W"]) < tol and relerr(out[2]["H"], out[4]["H"]) < tol
    assert not np.array_equal(out[2]["W"], out[4]["W"])


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_large_k_nan_and_fixed(ctx, dt):
    k = 40
    rng = np.random.default_rng(5)
    Xn = synth.mixture(300, 72, 4, seed=2, dtype=dt)
    Xn[rng.random(Xn.shape) < 0.15] = np.nan
    Xn[rng.random(Xn.shape) < 0.05] = 0.0
    W0, H0 = synth.philox_inits(5, 1, 300, k, 72, dtype=dt)
    tol = RTOL64 if dt == np.float64 else RTOL32
    Wt, Ht, ob = nb.trace(Xn, k, W0[0], H0[0], 12, ctx=ctx, engine=2)
    Wr, Hr = oracle_trace(Xn, k, W0[0], H0[0], 12)
    for t in (0, 1, 9, 11):
        assert relerr(Wt[t], Wr[t]) < tol and relerr(Ht[t], Hr[t]) < tol, t
    X = synth.mixture(300, 72, 4, seed=2, dtype=dt)
    for kw in ({"Wfixed": True}, {"Hfixed": True}):
        Wt, Ht, ob = nb.trace(X, k, W0[0], H0[0], 12, ctx=ctx, engine=2, **kw)
        Wr, Hr = oracle_trace(X, k, W0[0], H0[0], 12, **kw)
        assert relerr(Wt[-1], Wr[-1]) < tol and relerr(Ht[-1], Hr[-1]) < tol, kw


def test_large_k_rowsharded_single_rank():
    n, m, k, niter = 300, 64, 40, 12
    X = synth.mixture(n, m, 3, seed=7)
    W0, H0 = synth.philox_inits(11, 1, n, k, m)
    with nb.Context() as c:
        c.comm_init(1, 0, None, 0, n)
        Wt, Ht, ob = nb.trace(X, k, W0[0], H0[0], niter, ctx=c, engine=2)
    Wr, Hr = oracle_trace(X, k, W0[0], H0[0], niter)
    for t in range(niter):
        assert relerr(Wt[t], Wr[t]) < RTOL64, ("W", t)
        assert relerr(Ht[t], Hr[t]) < RTOL64, ("H", t)


def test_large_k_full_stop_rule_matches_oracle(ctx):
    """Default parameters (reference stop rule) at k = 36, which AUTO routes to the tiled engine: iteration counts, stop
    reasons, objective and normalised factors of every restart."""
    X = synth.mixture(120, 60, 3, seed=3)
    k, R = 36, 3
    W0, H0 = synth.philox_inits(100, R, 120, k, 60)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b])
    g = b.get()
    b.close()
    for r in range(R):
        inf = {}
        W, H, of = o.execute_singlerun_compute(X.copy(), k, Winit=W0[r].copy(), Hinit=H0[r].copy(), info=inf)
        assert g["iters"][r] == inf["iters"], (r, g["iters"][r], inf["iters"])
        assert g["stop_reason"][r] == {"maxiter": 1, "tol": 2, "reattempts": 3, "consistency": 4}[inf["stop_reason"]]
        assert g["obj_norm"][r] == pytest.approx(of, rel=1e-6, abs=1e-12)
        assert relerr(g["W"][r], W) < 1e-7 and relerr(g["H"][r], H) < 1e-7


def test_large_k_execute_across_32(ctx):
    """execute over k = 31..34: the resident engine below 33, the tiled engine above; kopt, robustness, fit, aic and the
    per-k factors against the oracle."""
    X = synth.mixture(90, 40, 3, seed=100)
    ks = range(31, 35)
    W, H, fit, rob, aic, kopt = nb.execute(X, ks, 4, seed=100, ctx=ctx, maxiter=150)
    Wo, Ho, fito, robo, aico, kopto = o.execute(X.copy(), ks, 4, seed=100, maxiter=150)
    assert kopt == kopto
    for k in ks:
        assert rob[k - 1] == pytest.approx(robo[k - 1], abs=1e-6), k
        assert fit[k - 1] == pytest.approx(fito[k - 1], rel=1e-5, abs=1e-10), k
        assert aic[k - 1] == pytest.approx(aico[k - 1], rel=1e-5), k
        assert relerr(W[k], Wo[k]) < 1e-6 and relerr(H[k], Ho[k]) < 1e-6, k


def test_large_k_normalizevector_and_cluster_wmatrix(ctx):
    n, m, k, R = 80, 50, 40, 6
    X = synth.mixture(n, m, 3, seed=8)
    nv = np.random.default_rng(1).random(n) + 0.5
    W0, H0 = synth.philox_inits(4, R, n, k, m)
    inits = [(W0[r].copy(), H0[r].copy()) for r in range(R)]
    Wg, Hg, fg, rg, ag = nb.execute_run(X, k, R, inits=(W0, H0), normalizevector=nv, maxiter=120, ctx=ctx)
    Wo, Ho, fo, ro, ao = o.execute_run(X.copy(order="F"), k, R, inits=inits, normalizevector=nv, maxiter=120)
    assert relerr(Wg, Wo) < 1e-7 and relerr(Hg, Ho) < 1e-7 and abs(fg - fo) <= 1e-7 * fo and abs(rg - ro) < 1e-8
    dg, do = {}, {}
    Wg, Hg, fg, rg, ag = nb.execute_run(X, k, R, inits=(W0, H0), clusterWmatrix=True, maxiter=120, ctx=ctx, details=dg)
    Wo, Ho, fo, ro, ao = o.execute_run(X.copy(), k, R, inits=inits, clusterWmatrix=True, maxiter=120, details=do)
    assert np.array_equal(dg["labels"], do["labels"]) and np.array_equal(dg["order"], do["idxsort"])
    assert relerr(Wg, Wo) < 1e-7 and relerr(Hg, Ho) < 1e-7
    assert abs(fg - fo) <= 1e-7 * fo and abs(rg - ro) < 1e-8 and abs(ag - ao) <= 1e-6 * abs(ao)
    assert np.allclose(dg["clustersil"], do["clustersil"][:, 0], atol=1e-9)


def test_large_k_clustering_many_restarts(ctx):
    """Clustering and silhouettes at k = 64 with 40 restarts: labels identical to the oracle on the solver's H stacks."""
    n, m, k, R = 150, 120, 64, 40
    X = synth.mixture(n, m, 3, seed=12)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.init_random(7)
    ctx.solve([b], nb.default_params(maxiter=30))
    g = b.get()
    cl = b.cluster()
    b.close()
    order = np.argsort(g["obj_norm"], kind="stable")
    assert list(cl["order"]) == list(order)
    Hs = [np.array(g["H"][i], dtype=np.float64) for i in order]
    Ws = [np.array(g["W"][i], dtype=np.float64) for i in order]
    labels, cent = o.clustersolutions(Hs, False)
    assert np.array_equal(cl["labels"], labels)
    _, _, csil, _, _ = o.finalize(Ws, Hs, labels, False)
    assert np.allclose(cl["clustersil"], csil[:, 0], atol=1e-9)
    assert np.allclose(cl["centroids"], cent, rtol=1e-10)


def test_large_k_refusals(ctx):
    X = synth.mixture(100, 40, 3, seed=1)
    ctx.set_X(X)
    b = ctx.batch(65, 1)
    b.init_random(1)
    with pytest.raises(nb.NMFkError) as e:
        ctx.solve([b])
    assert e.value.status == -6
    b.close()
    b = ctx.batch(40, 1)
    b.init_random(1)
    with pytest.raises(nb.NMFkError) as e:
        ctx.solve([b], nb.default_params(engine=1))
    assert e.value.status == -6
    b.close()
