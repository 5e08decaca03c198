"""GPU parity on the BASELINE.json configurations themselves (VERDICT r1 "next" #1): every case compares the CUDA path (through
the C ABI) with the CPU ORACLE - never with another engine of this repository.

  C2  1000 x 200 Float64      execute(X, 4:6, 10), full stop rule: iteration counts, stop reasons, labels, kopt (committed
                              oracle fixture tests/golden/c2_execute_k4_6.npz, made by tests/golden/make_c2_execute_golden.py)
  C3  10000 x 10000 Float32   k = 16, 2 restarts x 3 iterations through the tcgen05 pass            <= 1e-4
  C4  100000 x 2000 Float64   k = 32 / 5 / 3, 2 iterations through the DMMA / scalar tiled pass     <= 1e-9
  C5q 500000 x 1000 Float32   k = 24, 2 iterations (one quarter of C5: one GPU's share on 4 GPUs)   <= 1e-4
  clustering + silhouettes at R*k = 8000 rows (the size the 8-GPU sweep of C2 clusters), near-tie probe of the greedy argmin.
Tolerances are the north star's: 1e-9 relative (Float64), 1e-4 (Float32 against the Float64-computing reference)."""
import os

import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


def test_c2_execute_matches_oracle_golden(ctx):
    """BASELINE C2, execute(X, 4:6, 10) with the reference stop rule against the oracle fixture: identical iteration counts
    and stop reasons for all 30 restarts, identical sort order and cluster labels, robustness / fit / aic, kopt."""
    g = np.load(os.path.join(GOLDEN, "c2_execute_k4_6.npz"))
    X = synth.mixture(1000, 200, 5, seed=2015)
    for k in (4, 5, 6):
        det = {}
        W, H, fit, rob, aic = nb.execute_k(X, k, 10, seed=2015, ctx=ctx, details=det)
        assert np.array_equal(det["iters"], g["k%d_iters" % k]), (k, det["iters"], g["k%d_iters" % k])
        assert np.array_equal(det["order"], g["k%d_idxsort" % k]), k
        assert np.array_equal(det["labels"], g["k%d_labels" % k]), k
        assert np.allclose(det["fit"], g["k%d_objvalue" % k], rtol=1e-7, atol=1e-12), k
        assert np.allclose(det["clustersil"], g["k%d_clustersil" % k], atol=1e-8), k
        assert abs(rob - float(g["k%d_rob" % k])) < 1e-8
        assert abs(fit - float(g["k%d_fit" % k])) <= 1e-7 * float(g["k%d_fit" % k]) + 1e-12
        assert abs(aic - float(g["k%d_aic" % k])) <= 1e-6 * abs(float(g["k%d_aic" % k]))
        assert relerr(W, g["k%d_W" % k]) < 1e-6 and relerr(H, g["k%d_H" % k]) < 1e-6
    W, H, fit, rob, aic, kopt = nb.execute(X, range(4, 7), 10, seed=2015, ctx=ctx)
    kg = int(g["kopt"])
    assert kopt == (None if kg < 0 else kg)
    for k in (4, 5, 6):
        assert abs(float(rob[k - 1]) - float(g["k%d_rob" % k])) < 1e-8
    b = ctx.batch(5, 10)  # stop reasons of one k straight from the batch
    b.init_random(2015)
    ctx.solve([b])
    st = b.get(factors=False)
    b.close()
    assert np.array_equal(st["stop_reason"], g["k5_stop"]) and np.array_equal(st["iters"], g["k5_iters"])


def _fixed_iterations_vs_oracle(ctx, n, m, k0, k, R, niter, dt, tol, engine=2):
    X = synth.mixture(n, m, k0, seed=2015, dtype=dt)
    W0, H0 = synth.philox_inits(2015, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(maxiter=niter, engine=engine, normalize=0))
    out = b.get()
    b.close()
    X64 = np.asfortranarray(X.astype(np.float64))
    for r in range(R):
        W, H, obj = o.nmf_multiplicative(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=niter)
        eW, eH = relerr(out["W"][r], W), relerr(out["H"][r], H)
        assert eW < tol and eH < tol, (r, eW, eH)
        assert abs(out["obj_ssq"][r] - obj) <= (1e-7 if dt == np.float64 else 2e-3) * obj + 1e-12, (r, out["obj_ssq"][r], obj)
        assert out["iters"][r] == niter


def test_c3_shape_tcgen05_pass_vs_oracle(ctx):
    """BASELINE C3 (10000 x 10000 Float32, k = 16): 2 restarts x 3 iterations of the tcgen05 tiled pass against the Float64
    oracle from the same initial factors."""
    _fixed_iterations_vs_oracle(ctx, 10000, 10000, 16, 16, 2, 3, np.float32, 1e-4)


def test_c3_variant_fro_vs_oracle(ctx, capfd):
    """C3 through Variant FRO as bench.py runs it (10000 x 10000 Float32 mixture, k = 16, 64 restarts, Philox initial factors):
    3 iterations of the stacked solve, which runs the cluster-multicast GEMM over 8 M tiles with 6 / 6 split-K slices and the
    Gram sums in 4 / 4 slices.  Restarts 0 (first tile), 8 (second tile, the second CTA of a cluster), 15 (holds row 255, the
    last row of a cluster pair) and 63 (last tile) against the Float64 oracle."""
    n, m, k, R, niter = 10000, 10000, 16, 64, 3
    X = synth.mixture(n, m, 16, seed=2015, dtype=np.float32)
    W0, H0 = synth.philox_inits(2015, R, n, k, m, dtype=np.float32)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(variant=1, maxiter=niter, normalize=0))
    out = b.get()
    b.close()
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1)
    X64 = X.astype(np.float64)
    del X
    delta = float(np.sqrt(np.finfo(np.float32).eps))
    for r in (0, 8, 15, 63):
        W, H, _ = o.nmf_multupdate_mse(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=niter, tol=0.0,
                                       delta=delta)
        eW, eH = relerr(out["W"][r], W), relerr(out["H"][r], H)
        assert eW < 1e-4 and eH < 1e-4, (r, eW, eH)
    err = capfd.readouterr().err
    assert "barrier time-out" not in err, err[-2000:]


@pytest.mark.parametrize("k", [32, 5, 3])
def test_c4_shape_tiled_pass_vs_oracle(ctx, k):
    """BASELINE C4 (100000 x 2000 Float64): k = 32 and 5 run the DMMA tiled pass, k = 3 the scalar-FMA pass."""
    _fixed_iterations_vs_oracle(ctx, 100000, 2000, 8, k, 1, 2, np.float64, 1e-9)


def test_c5_quarter_shape_tcgen05_pass_vs_oracle(ctx):
    """One GPU's share of BASELINE C5 on 4 GPUs (500000 x 1000 Float32, k = 24): 2 iterations against the oracle."""
    _fixed_iterations_vs_oracle(ctx, 500000, 1000, 24, 24, 1, 2, np.float32, 1e-4)


def test_float32_execute_decisions_vs_oracle(ctx):
    """Float32 execute through the tcgen05 tiled engine against the Float64-computing oracle (SURVEY 0.4) on a 3-source
    mixture with margin: identical kopt, identical robustness decisions, identical cluster labels at the well-determined k,
    and iteration counts within the honest tolerance - the stop machine compares objective changes with tolOF = 1e-3 on
    Float32-rounded factors, so a check can fall on the other side of the threshold: at most 2 check periods (20 iterations)
    apart for every restart."""
    X = synth.mixture(1200, 400, 3, seed=31, dtype=np.float32)
    ks, R = [2, 3, 4], 6
    robs_g, robs_o = {}, {}
    for k in ks:
        W0, H0 = synth.philox_inits(77, R, 1200, k, 400, dtype=np.float32)
        dg, do = {}, {}
        Wg, Hg, fg, rg, ag = nb.execute_run(X, k, R, inits=(W0, H0), ctx=ctx, engine=2, maxiter=400, details=dg)
        Wo, Ho, fo, ro, ao = o.execute_run(np.asfortranarray(X.copy()), k, R, inits=[(W0[r].copy(), H0[r].copy()) for r in range(R)],
                                           maxiter=400, details=do)
        robs_g[k], robs_o[k] = float(rg), float(ro)
        di = np.abs(dg["iters"].astype(int) - do["iters"].astype(int))
        assert di.max() <= 20, (k, dg["iters"], do["iters"])
        assert abs(fg - fo) <= 2e-3 * fo + 1e-6, (k, fg, fo)
        if k <= 3:
            assert np.array_equal(dg["order"], do["idxsort"]), k
            assert np.array_equal(dg["labels"], do["labels"]), k
            assert abs(rg - ro) < 5e-3, (k, rg, ro)
            assert relerr(Wg, Wo) < 5e-3 and relerr(Hg, Ho) < 5e-3
    assert [robs_g[k] > 0.5 for k in ks] == [robs_o[k] > 0.5 for k in ks]
    kg = nb.getk(ks, [robs_g[k] for k in ks])
    assert kg == o.getk(ks, [robs_o[k] for k in ks]) == 3


def _random_solutions(rng, R, k, m, noise):
    base = rng.random((k, m)) ** 3
    H = np.empty((R, k, m))
    for r in range(R):
        H[r] = base[rng.permutation(k)] * (1 + noise * rng.standard_normal((k, m)))
    H = np.abs(H)
    H /= H.sum(axis=2, keepdims=True)
    return H, rng.random(R)


def test_clustering_at_8000_rows_vs_oracle(ctx):
    """clustersolutions + finalize silhouettes at R*k = 8000 (R_total = 800 solutions of k = 10, the size the 8-GPU sweep of C2
    clusters): labels bit-identical, silhouettes <= 1e-9."""
    rng = np.random.default_rng(8)
    R, k, m = 800, 10, 200
    H, obj = _random_solutions(rng, R, k, m, 0.05)
    ctx.set_X(synth.mixture(50, m, 3, seed=1))
    b = ctx.import_solutions(H, obj)
    cl = b.cluster()
    b.close()
    order = np.argsort(obj, kind="stable")
    assert np.array_equal(cl["order"], order)
    Hs = [H[i] for i in order]
    labels, cent = o.clustersolutions(Hs, False)
    assert np.array_equal(cl["labels"], labels)
    _, _, csil, _, _ = o.finalize([np.zeros((1, k))] * R, Hs, labels, False)
    assert np.allclose(cl["clustersil"], csil[:, 0], atol=1e-9)
    assert np.allclose(cl["centroids"], cent, rtol=1e-10)


def test_greedy_argmin_ties_break_like_the_reference(ctx):
    """Exact ties in the k x k distance matrix of clustersolutions (duplicate rows inside a solution): `argmin` takes the first
    minimum in column-major order (NMFkCluster.jl:476) - the device must take the same one."""
    rng = np.random.default_rng(3)
    k, m, R = 4, 16, 9
    H = rng.integers(1, 9, (R, k, m)).astype(np.float64)  # small integers: dot products are exact in any summation order
    H[:, 1] = H[:, 0]  # rows 0 and 1 of every solution are identical -> equal columns of D
    H[2, 3] = H[2, 2]
    obj = np.arange(R, dtype=np.float64)
    ctx.set_X(synth.mixture(20, m, 2, seed=1))
    b = ctx.import_solutions(H, obj)
    cl = b.cluster()
    b.close()
    labels, _ = o.clustersolutions([H[i] for i in range(R)], False)
    assert np.array_equal(cl["labels"], labels)
