"""Variant KL_DIV (method=:nmf, algorithm=:multmse -> NMF.MultUpdate(obj=:div)) on the tiled engine against the
restatement of NMF.jl in tests/test_oracle_multmse_cpu.py (nmf_multupdate_div): per-iteration factors through every pass kernel, the
benchmark matrices, the stop rule, exact zeros, pause / resume, restart batches, execute_run / execute, and the refusals.
Tolerances: 1e-9 relative for Float64, 1e-4 for Float32, against the Float64 oracle with the delta of the data type."""
import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o
from test_oracle_multmse_cpu import execute_singlerun_nmf_multmse, multupdate_div_delta, nmf_multupdate_div

pytestmark = pytest.mark.gpu
KL_DIV = 3


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


def _trace(ctx, X, k, W0, H0, niter, **kw):
    """W, H of every restart after each of the first niter iterations (paused runs, iter_limit = t)."""
    ctx.set_X(X)
    b = ctx.batch(k, W0.shape[0])
    b.set_init(W0, H0)
    outs = []
    for t in range(1, niter + 1):
        ctx.solve([b], nb.default_params(variant=KL_DIV, maxiter=10 ** 6, iter_limit=t, normalize=0, tol=0.0, **kw))
        g = b.get()
        outs.append((g["W"].copy(), g["H"].copy()))
    b.close()
    return outs


def _oracle_trace(X, k, W0, H0, niter, dt):
    ref = []
    nmf_multupdate_div(X.astype(np.float64), k, Winit=W0.astype(np.float64), Hinit=H0.astype(np.float64), maxiter=niter, tol=0.0,
                       delta=multupdate_div_delta(dt), trace=lambda it, W, H: ref.append((W.copy(), H.copy())))
    return ref


def _check(outs, X, k, W0, H0, niter, dt, restarts):
    tol = 1e-9 if dt == np.float64 else 1e-4
    for r in restarts:
        ref = _oracle_trace(X, k, W0[r], H0[r], niter, dt)
        for t in range(niter):
            assert relerr(outs[t][0][r], ref[t][0]) < tol, ("W", r, t, relerr(outs[t][0][r], ref[t][0]))
            assert relerr(outs[t][1][r], ref[t][1]) < tol, ("H", r, t, relerr(outs[t][1][r], ref[t][1]))


# pass kernel reached by each case (solve_tiled_t): Float32 with n, m multiples of 4 -> tcgen05 (tc2_pass_kernel for k <= 16,
# tc_pass_kernel above); Float64 with k >= 4 -> tiled_dmma_pass_kernel; Float32 with n or m not a multiple of 4, Float64 with
# k < 4, and engine = TILED_SCALAR -> tiled_pass_kernel
CASES = [  # n, m, k, R, dt, engine, pass
    (1024, 768, 8, 5, np.float32, 0, "tc2"), (2048, 512, 16, 6, np.float32, 0, "tc2"),
    (1024, 768, 20, 3, np.float32, 0, "tc"), (768, 1024, 48, 2, np.float32, 0, "tc"), (512, 640, 64, 2, np.float32, 0, "tc"),
    (1000, 600, 4, 3, np.float64, 0, "dmma"), (700, 900, 32, 3, np.float64, 0, "dmma"), (600, 500, 64, 2, np.float64, 0, "dmma"),
    (1001, 603, 8, 3, np.float32, 0, "scalar"), (800, 500, 3, 3, np.float64, 0, "scalar"),
    (1024, 768, 12, 3, np.float32, 4, "scalar"), (900, 700, 24, 2, np.float64, 4, "scalar"),
]


@pytest.mark.parametrize("n,m,k,R,dt,engine,kind", CASES, ids=["%s-%s-k%d" % (c[6], np.dtype(c[4]).name, c[2]) for c in CASES])
def test_per_iteration_vs_oracle(ctx, n, m, k, R, dt, engine, kind):
    X = synth.mixture(n, m, 5, seed=11 + k, dtype=dt)
    W0, H0 = synth.philox_inits(31 + k, R, n, k, m, dtype=dt)
    niter = 6
    outs = _trace(ctx, X, k, W0, H0, niter, engine=engine)
    _check(outs, X, k, W0, H0, niter, dt, range(R))


def test_c3_matrix_64_restarts(ctx):
    """The C3 matrix (10000 x 10000 Float32, k = 16, 64 restarts: tc2_pass_kernel with 16 restart groups) for three iterations;
    restarts 0, 31 and 63 against the oracle."""
    n = m = 10000
    k, R = 16, 64
    X = synth.mixture(n, m, 16, seed=2015, dtype=np.float32)
    W0, H0 = synth.philox_inits(5, R, n, k, m, dtype=np.float32)
    outs = _trace(ctx, X, k, W0, H0, 3)
    _check(outs, X, k, W0, H0, 3, np.float32, [0, 31, 63])


def test_c4_matrix_k32(ctx):
    """The C4 matrix (100000 x 2000 Float64) at k = 32 with 4 restarts (tiled_dmma_pass_kernel, sliced H-update), two iterations."""
    n, m, k, R = 100000, 2000, 32, 4
    X = synth.mixture(n, m, 8, seed=4, dtype=np.float64)
    W0, H0 = synth.philox_inits(8, R, n, k, m)
    outs = _trace(ctx, X, k, W0, H0, 2)
    _check(outs, X, k, W0, H0, 2, np.float64, [0, R - 1])


@pytest.mark.parametrize("dt,engine", [(np.float64, 0), (np.float64, 4), (np.float32, 0)])
def test_stop_rule_and_execute_singlerun(ctx, dt, engine):
    """NMF.jl stop_condition with a loose tol: the iteration count of the oracle and stop reason 2 (Float64; in Float32 the
    count may differ by rounding, the factors still match); objective = normnan(X - W*H), rows of H sum to one."""
    n, m, k, R = 400, 120, 3, 4
    X = synth.mixture(n, m, 3, seed=5, dtype=dt)
    W0, H0 = synth.philox_inits(9, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(variant=KL_DIV, maxiter=5000, tol=1e-4, engine=engine))
    g = b.get()
    b.close()
    tol = 1e-7 if dt == np.float64 else 1e-3
    for r in range(R):
        inf = {}
        W, H, obj = execute_singlerun_nmf_multmse(X.astype(np.float64), k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64),
                                                  maxiter=5000, tol=1e-4, info=inf, delta=multupdate_div_delta(dt))
        assert inf["converged"] and inf["iters"] < 5000
        if dt == np.float64:
            assert g["iters"][r] == inf["iters"] and g["stop_reason"][r] == 2, (r, g["iters"][r], inf)
            assert relerr(g["W"][r], W) < tol and relerr(g["H"][r], H) < tol
            assert abs(g["obj_norm"][r] - obj) <= tol * obj
        else:
            assert g["stop_reason"][r] == 2 and abs(int(g["iters"][r]) - inf["iters"]) <= 0.05 * inf["iters"] + 2, (g["iters"][r], inf)
        assert np.allclose(g["H"][r].sum(axis=1), 1.0, atol=1e-5 if dt == np.float32 else 1e-12)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_exact_zeros_objective_on_restored_x(ctx, dt):
    """Exact zeros of X (two whole columns and scattered entries): factors against the oracle, which uses X as given, and the
    objective normnan(X - W*H) against the X with its zeros."""
    n, m, k, R, it = 640, 480, 6, 3, 7
    X = synth.mixture(n, m, 4, seed=13, dtype=dt)
    rng = np.random.default_rng(1)
    X[rng.random((n, m)) < 0.2] = 0
    X[:, [3, 100]] = 0
    W0, H0 = synth.philox_inits(17, R, n, k, m, dtype=dt)
    outs = _trace(ctx, X, k, W0, H0, it)
    _check(outs, X, k, W0, H0, it, dt, range(R))
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(variant=KL_DIV, maxiter=it, tol=0.0))
    g = b.get()
    b.close()
    tol = 1e-9 if dt == np.float64 else 1e-4
    for r in range(R):
        W, H, obj = execute_singlerun_nmf_multmse(X.astype(np.float64), k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64),
                                                  maxiter=it, tol=0.0, delta=multupdate_div_delta(dt))
        assert g["stop_reason"][r] == 1 and g["iters"][r] == it
        assert abs(g["obj_norm"][r] - obj) <= tol * obj, (r, g["obj_norm"][r], obj)


@pytest.mark.parametrize("dt,n,m,k", [(np.float64, 1500, 700, 12), (np.float32, 2048, 1024, 16), (np.float32, 1024, 512, 40)])
def test_resume_equals_continuous_and_restart_alone(ctx, dt, n, m, k):
    """Runs paused every 7 iterations and resumed equal the continuous run; restart 2 solved alone equals restart 2 of the batch
    (Float64 bit for bit, Float32 <= 2e-5)."""
    R, total = 5, 30
    X = synth.mixture(n, m, 5, seed=21, dtype=dt)
    W0, H0 = synth.philox_inits(3, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    p = dict(variant=KL_DIV, maxiter=total, tol=0.0, normalize=0)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(**p))
    cont = b.get()
    b.set_init(W0, H0)
    for lim in range(7, total + 7, 7):
        ctx.solve([b], nb.default_params(iter_limit=min(lim, total), **p))
    res = b.get()
    b.close()
    assert np.array_equal(cont["W"], res["W"]) and np.array_equal(cont["H"], res["H"])
    assert list(cont["iters"]) == list(res["iters"]) == [total] * R
    one = ctx.batch(k, 1)
    one.set_init(W0[2:3], H0[2:3])
    ctx.solve([one], nb.default_params(**p))
    g1 = one.get()
    one.close()
    if dt == np.float64:
        assert np.array_equal(g1["W"][0], cont["W"][2]) and np.array_equal(g1["H"][0], cont["H"][2])
    else:
        assert relerr(g1["W"][0], cont["W"][2]) <= 2e-5 and relerr(g1["H"][0], cont["H"][2]) <= 2e-5


def test_execute_run_and_execute(ctx):
    """execute_run / execute with method="nmf", algorithm="multmse": fit, robustness and kopt from the oracle's solver composed
    with clustersolutions / finalize (the decisions of execute_run), rows of H sum to one."""
    X = synth.mixture(400, 120, 3, seed=5)
    R, maxiter = 6, 200
    fits, robs = [], []
    for k in (2, 3, 4):
        W0, H0 = synth.philox_inits(40 + k, R, 400, k, 120)
        Wg, Hg, fg, rg, ag = nb.execute_run(X, k, R, inits=(W0, H0), method="nmf", algorithm="multmse", maxiter=maxiter, tol=0.0, ctx=ctx)
        sols = [execute_singlerun_nmf_multmse(X.copy(), k, Winit=W0[r].copy(), Hinit=H0[r].copy(), maxiter=maxiter, tol=0.0)
                for r in range(R)]
        order = np.argsort([s[2] for s in sols], kind="stable")
        assert abs(fg - sols[order[0]][2]) <= 1e-7 * sols[order[0]][2]
        labels, _ = o.clustersolutions([sols[i][1] for i in order], False)
        _, _, csil, _, _ = o.finalize([sols[i][0] for i in order], [sols[i][1] for i in order], labels, False)
        assert abs(rg - float(csil.min())) < 1e-7
        assert np.allclose(Hg.sum(axis=1), 1.0, atol=1e-9)
        fits.append(fg)
        robs.append(rg)
    inits = {k: synth.philox_inits(40 + k, R, 400, k, 120) for k in (2, 3, 4)}
    W, H, fit, rob, aic, kopt = nb.execute(X, [2, 3, 4], R, inits=inits, method="nmf", algorithm="multmse", maxiter=maxiter, tol=0.0,
                                           ctx=ctx)
    assert np.allclose(np.asarray(fit[1:], dtype=float), fits, rtol=1e-7) and np.allclose(np.asarray(rob[1:], dtype=float), robs, atol=1e-7)
    assert kopt == o.getk([2, 3, 4], robs)
    with pytest.raises(nb.NMFkError):
        nb.execute_run(X, 3, R, method="nmf", algorithm="alspgrad", ctx=ctx)


def test_refusals(ctx):
    X = synth.mixture(200, 100, 3, seed=2)
    W0, H0 = synth.philox_inits(1, 2, 200, 3, 100)

    def solve(k=3, Xs=X, W=W0, H=H0, **kw):
        b = ctx.batch(k, 2)
        try:
            b.set_init(W, H)
            ctx.solve([b], nb.default_params(variant=KL_DIV, maxiter=5, **kw))
        finally:
            b.close()

    ctx.set_X(X)
    for kw in (dict(stop_rule=1), dict(engine=1), dict(engine=3)):
        with pytest.raises(nb.NMFkError, match="KL_DIV"):
            solve(**kw)
    W65, H65 = synth.philox_inits(1, 2, 200, 65, 100)
    with pytest.raises(nb.NMFkError, match="KL_DIV"):
        solve(k=65, W=W65, H=H65)
    ctx.set_X(X, normalizevector=np.full(200, 2.0))
    with pytest.raises(nb.NMFkError, match="KL_DIV"):
        solve()
    ctx.set_X(X)
    ctx.set_weight(np.linspace(0.5, 1.5, 200))
    with pytest.raises(nb.NMFkError, match="KL_DIV"):
        solve()
    ctx.set_weight(None)
    Xn = X.copy()
    Xn[3, 4] = np.nan
    ctx.set_X(Xn)
    with pytest.raises(nb.NMFkError, match="KL_DIV"):
        solve()
    solo = nb.Context()
    try:
        solo.comm_init(1, 0, None, 0, 200)
        solo.set_X(X)
        b = solo.batch(3, 2)
        b.set_init(W0, H0)
        with pytest.raises(nb.NMFkError, match="KL_DIV"):
            solo.solve([b], nb.default_params(variant=KL_DIV, maxiter=5))
        b.close()
    finally:
        solo.close()
