"""Pins the CPU oracle against every known answer the reference holds for this path
(SURVEY.md §8c).  CPU-only."""
import os

import numpy as np
import pytest

from oracle import nmfk_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))


def bss_X():
    return np.loadtxt(os.path.join(HERE, "golden", "bss_notebook_X.csv"), delimiter=",")


def test_bss_notebook_recorded_outputs():
    """notebooks/blind_source_separation/blind_source_separation.md:230-264 (reference's own
    recorded run on the printed X): k=2 Fit 13.93858 (sum of squares in that NMFk version),
    silhouette 0.994, AIC -46.21 (with phi = SSQ), kopt = 3, silhouette(4),(5) < 0.5."""
    X = bss_X()
    W, H, fit, rob, aic, kopt = o.execute(X, range(2, 6), 10, seed=2021)
    assert kopt == 3
    assert fit[1] ** 2 == pytest.approx(13.93858, rel=2e-3)
    assert rob[1] > 0.95 and rob[2] > 0.5 and rob[3] < 0.5 and rob[4] < 0.5
    # AIC formula of NMFkExecute.jl:708 evaluated with the notebook's phi (= SSQ there)
    n, m = X.shape
    assert 2 * (n * 2 + 2 * m) + n * m * np.log(13.93858 / (n * m)) == pytest.approx(-46.21209, abs=1e-4)
    # and with this version's phi (= norm) it is what the oracle returns
    assert aic[1] == pytest.approx(2 * (n * 2 + 2 * m) + n * m * np.log(fit[1] / (n * m)), rel=1e-12)
    assert fit[2] < 0.1 and fit[3] < 0.1 and fit[4] < 0.1  # rank-3 data: k >= 3 fits


def test_readme_example_kopt_is_3():
    """Readme.md:97-131: a,b,c ~ U(0,1)^15, X = [a+3c, 10a+b, b, 5b+c, a+2b+5c] -> kopt = 3,
    silhouette(2),(3) > 0.5 > silhouette(4),(5)."""
    rng = np.random.Generator(np.random.Philox(key=2015))
    a, b, c = rng.random(15), rng.random(15), rng.random(15)
    X = np.stack([a + 3 * c, 10 * a + b, b, 5 * b + c, a + 2 * b + 5 * c], axis=1)
    W, H, fit, rob, aic, kopt = o.execute(X, range(2, 6), 10, seed=100)
    assert kopt == 3
    assert rob[1] > 0.5 and rob[2] > 0.5 and rob[3] < 0.5 and rob[4] < 0.5
    assert fit[0] == np.inf and rob[0] == -1  # NMFkExecute.jl:200-201


def test_feature_extraction_kopt_is_4():
    """notebooks/feature_extraction/feature_extraction.jl:10-24 + .md:208-292: three sines + one
    random signal mixed by a fixed 4x10 H -> silhouettes high for k<=4, negative after, kopt=4.
    (s4 comes from Julia's RNG there; drawn from Philox here.)  Range trimmed to 2:6 for time."""
    t = np.arange(1, 101)
    s1 = (np.sin(0.05 * t) + 1) / 2
    s2 = (np.sin(0.3 * t) + 1) / 2
    s3 = (np.sin(0.5 * t) + 1) / 2
    s4 = np.random.Generator(np.random.Philox(key=2021)).random(100)
    W0 = np.stack([s1, s2, s3, s4], axis=1)
    H0 = np.array([[1, 5, 0, 0, 1, 1, 2, 1, 0, 2], [0, 1, 1, 5, 2, 1, 0, 0, 2, 3], [3, 0, 0, 1, 0, 1, 0, 5, 4, 3],
                   [1, 1, 4, 1, 5, 0, 1, 1, 5, 3]], dtype=float)
    X = W0 @ H0
    W, H, fit, rob, aic, kopt = o.execute(X, range(2, 7), 10, seed=7)
    assert kopt == 4
    assert rob[3] > 0.9 and rob[4] < 0.5 and rob[5] < 0.5
    # recovered H(k=4) rows sum to one (test_execute_smoke.jl:18-19) and match the
    # row-normalised true H up to a permutation (Hmatrix-4.csv in the notebook directory)
    He = H[4]
    assert np.allclose(He.sum(axis=1), 1.0, atol=1e-4)
    Hn = H0 / H0.sum(axis=1, keepdims=True)
    for row in Hn:
        assert min(np.abs(He - row).max(axis=1)) < 5e-2


def test_execute_smoke_invariants():
    """test/test_execute_smoke.jl:6-32."""
    rng = np.random.default_rng(123)
    X = np.abs(rng.standard_normal((5, 4)))
    X0 = X.copy()
    W, H, obj = o.execute_singlerun_compute(X, 2, maxiter=50, tol=1e-8, rng=np.random.default_rng(1))
    assert W.shape == (5, 2) and H.shape == (2, 4)
    assert np.isfinite(obj) and np.isfinite(W).all() and np.isfinite(H).all()
    assert (W >= 0).all() and (H >= 0).all()
    assert H[0].sum() == pytest.approx(1.0, abs=1e-4) and H[1].sum() == pytest.approx(1.0, abs=1e-4)
    assert np.array_equal(X, X0)  # caller's X restored (NMFkMultiplicative.jl:123-124)
    X = np.abs(np.random.default_rng(321).standard_normal((6, 5)))
    Wa, Ha, phi, minsil, aic = o.execute_run(X, 1, 2, maxiter=40, tol=1e-8, seed=3)
    assert Wa.shape == (6, 1) and Ha.shape == (1, 5)
    assert np.isfinite(phi) and np.isfinite(aic) and minsil == 1


def test_clustersolutions_unit():
    """test/test_cluster_unit.jl:36-54."""
    f1 = np.array([[1.0, 0], [0, 1], [1, 0], [0, 1]])
    f2 = np.array([[0.0, 1], [1, 0], [0, 1], [1, 0]])
    labels, centers = o.clustersolutions([f1, f2], True)
    assert labels.shape == (2, 2)
    assert list(labels[:, 0]) == [1, 2]
    assert sorted(labels[:, 1]) == [1, 2]
    assert list(labels[:, 1]) == [2, 1]
    assert centers.shape == (2, 4)


def test_helpers_known_answers():
    """test/test_normalize.jl:44-55 (zerostoepsilon floor eps(Float64)^2) and
    test/test_helpers.jl:60-67 (NaN-ignoring sums of squares)."""
    x = np.array([0.0, 1e-40, 1.0, -1.0])
    y = o.zerostoepsilon(x)
    e = np.finfo(np.float64).eps ** 2
    assert y[0] == e and y[1] == e and y[2] == 1.0 and y[3] == e
    assert x[0] == 0.0  # copy
    assert o.zerostoepsilon(np.zeros(2, dtype=np.float32))[0] == np.float32(np.finfo(np.float32).eps) ** 2
    t = np.array([1.0, np.nan, 3.0])
    assert o.ssqrnan(t - np.array([1.0, 5.0, 2.0])) == 1.0
    assert o.normnan(np.array([3.0, np.nan, 4.0])) == 5.0


def test_getk_and_signalorder():
    """src/NMFkPostprocess.jl:7-41,148-158."""
    assert o.getk([2, 3, 4, 5], [0.99, 0.85, -0.57, -0.67]) == 3
    assert o.getk([2, 3, 4], [0.1, 0.2, 0.3]) is None
    assert o.getk([2, 3, 4], [0.1, 0.2, 0.3], strict=False) == 4
    assert o.getk([2, 3], [np.nan, np.nan]) == 0
    assert o.getk([3], [0.6]) == 3 and o.getk([3], [0.4]) is None
    assert o.getk([2, 3, 4], [0.9, 0.2, 0.7]) == 4  # findlast, not "first drop"
    W = np.array([[1.0, 2.0], [1.0, 2.0]])
    H = np.array([[1.0, 1.0], [3.0, 3.0]])
    assert list(o.signalorder(W, H)) == [1, 0]


def test_negative_entries_raise_and_nan_quirk():
    """NMFkMultiplicative.jl:4-7; minimum() propagates NaN so NaN + negative passes."""
    with pytest.raises(o.NegativeEntriesError):
        o.nmf_preprocessing(np.array([[1.0, -1.0]]))
    inan, izero = o.nmf_preprocessing(np.array([[np.nan, -1.0, 0.0, 2.0]]))
    assert list(inan[0]) == [True, False, False, False] and list(izero[0]) == [False, True, True, False]


def test_silhouettes_against_sklearn():
    """Clustering.silhouettes restatement == textbook silhouette on a precomputed metric."""
    from sklearn.metrics import silhouette_samples
    rng = np.random.default_rng(0)
    V = rng.random((30, 6))
    D = o.pairwise_cosine_rows(V)
    lab = np.tile(np.arange(1, 4), 10)
    s = o.silhouettes(lab, D)
    ref = silhouette_samples(D, lab, metric="precomputed")
    assert np.allclose(s, ref, atol=1e-12)
    from scipy.spatial.distance import cdist
    assert np.allclose(D, cdist(V, V, "cosine"), atol=1e-12)


def test_finalize_means_and_variances_hand_case():
    """finalize (NMFkFinalize.jl:68-74): per-cluster mean / corrected variance over the trials of the member the labels
    pick, on a case small enough to do by hand; best=false of execute_run returns exactly these means."""
    import numpy as np
    from oracle import nmfk_oracle as o
    # 3 trials, k = 2: trial 2 has its rows swapped with respect to the clusters
    H = [np.array([[1.0, 2.0], [10.0, 20.0]]), np.array([[30.0, 40.0], [3.0, 4.0]]), np.array([[5.0, 6.0], [50.0, 60.0]])]
    W = [np.array([[1.0, 100.0]]), np.array([[300.0, 3.0]]), np.array([[5.0, 500.0]])]
    idx = np.array([[1, 2, 1], [2, 1, 2]])  # labels[a, t]
    Wm, Hm, csil, Wv, Hv = o.finalize(W, H, idx, False)
    assert np.allclose(Hm, [[3.0, 4.0], [30.0, 40.0]])
    assert np.allclose(Wm, [[3.0, 300.0]])
    assert np.allclose(Hv, [[4.0, 4.0], [400.0, 400.0]])  # var([1,3,5]) = 4, var([10,30,50]) = 400 (corrected)
    assert np.allclose(Wv, [[4.0, 40000.0]])
    assert csil.shape == (2, 1)


# ---------------------------------------------------------------------------------------------------------------------
# round 2: the restated third-party pieces next to the path (NMF.jl MultUpdate, Clustering.kmeans, sortclustering) and the
# reference-behaviour details the oracle mirrors (clusterWmatrix aliasing, DArray stop rule, Julia weight broadcasting)
# ---------------------------------------------------------------------------------------------------------------------
def test_fro_oracle_is_the_lee_seung_frobenius_update():
    """NMF.jl MultUpdate(obj=:mse): the Frobenius objective never increases (Lee & Seung 2001, theorem 1; delta only damps
    the step) and a rank-3 mixture is recovered."""
    rng = np.random.default_rng(0)
    X = rng.random((40, 3)) @ rng.random((3, 25))
    W0, H0 = rng.random((40, 3)), rng.random((3, 25))
    objs = []
    o.nmf_multupdate_mse(X, 3, Winit=W0, Hinit=H0, maxiter=300, tol=0.0, trace=lambda it, W, H: objs.append(float(np.sum((X - W @ H) ** 2))))
    assert all(b <= a * (1 + 1e-12) for a, b in zip(objs, objs[1:]))
    assert objs[-1] < 1e-3 * objs[0]
    inf = {}
    o.nmf_multupdate_mse(X, 3, Winit=W0, Hinit=H0, maxiter=100000, tol=1e-3, info=inf)
    assert inf["converged"] and inf["iters"] < 100000  # stop_condition: relative change of every column / row below tol


def test_darray_rule_equals_dense_rule_until_the_dense_one_gives_up():
    X = np.asfortranarray(np.random.default_rng(1).random((12, 3)) @ np.random.default_rng(2).random((3, 6)))
    W0, H0 = np.random.default_rng(3).random((12, 3)), np.random.default_rng(4).random((3, 6))
    i1 = {}
    Wd, Hd, _ = o.nmf_multiplicative(X.copy(), 3, Winit=W0.copy(), Hinit=H0.copy(), maxiter=40, info=i1)
    Wa, Ha, _ = o.nmf_multiplicative_darray(X.copy(), 3, Winit=W0.copy(), Hinit=H0.copy(), maxiter=40)
    assert i1["iters"] == 40 and np.allclose(Wd, Wa, rtol=1e-13) and np.allclose(Hd, Ha, rtol=1e-13)


def test_julia_weight_broadcasting():
    w = o._julia_weight(np.arange(4.0), 4, 3)
    assert w.shape == (4, 1)  # a Vector weights the ROWS
    assert o._julia_weight(np.ones((1, 3)), 4, 3).shape == (1, 3) and o._julia_weight(2.0, 4, 3) == 2.0


def test_cluster_wmatrix_aliases_the_best_solution():
    """clustersolutions(W stack, true) accumulates the centroids IN factors[1] (NMFkCluster.jl:453-455, :484, :512)."""
    rng = np.random.default_rng(5)
    Ws = [rng.random((7, 2)) + 0.1 for _ in range(4)]
    first = Ws[0].copy()
    labels, cent = o.clustersolutions(Ws, True)
    assert not np.array_equal(Ws[0], first) and np.allclose(Ws[0], cent.T)  # the caller's matrix now holds the centroids
    Hs = [rng.random((2, 7)) + 0.1 for _ in range(4)]
    keep = [h.copy() for h in Hs]
    o.clustersolutions(Hs, False)
    assert all(np.array_equal(a, b) for a, b in zip(Hs, keep))  # permutedims copies: nothing is aliased on the H branch


def test_kmeans_lloyd_and_sortclustering():
    rng = np.random.default_rng(6)
    X = np.hstack([np.array([[1.0], [0.1]]) + 0.01 * rng.random((2, 3)), np.array([[0.1], [1.0]]) + 0.01 * rng.random((2, 7))])
    r = o.kmeans_lloyd(X, 2, [0, 9])
    assert r["converged"] and sorted(r["counts"].tolist()) == [3, 7] and r["totalcost"] < 1e-3
    s = o.sortclustering(r)
    assert list(s["counts"]) == [7, 3] and list(s["assignments"][:3]) == [2, 2, 2] and list(s["assignments"][3:]) == [1] * 7
    res, sil = o.robustkmeans(X, 2, [[0, 1], [0, 9], [3, 4]], compute_silhouettes_flag=True)
    assert list(res["counts"]) == [7, 3] and sil.min() > 0.9


def test_execute_run_filters_follow_the_reference_index_mix():
    X = np.asfortranarray(np.random.default_rng(7).random((10, 2)) @ np.random.default_rng(8).random((2, 6)))
    det = {}
    o.execute_run(X.copy(), 2, 5, seed=3, maxiter=50, acceptratio=0.6, details=det)
    assert det["idxsol"].tolist() == [True, True, True, False, False] and det["labels"].shape == (2, 3)


def test_nmfsparsity_oracle_properties():
    """NMFsparsity (NMFkSparsity.jl): W keeps unit-norm columns (:86); with sparsity = 0 and beta = 2 the Euclidean divergence of
    the clamped model never increases; the L1 penalty shrinks sum(H)."""
    rng = np.random.default_rng(11)
    X = rng.random((30, 3)) @ rng.random((3, 20)) + 0.01
    W0, H0 = rng.random((30, 3)), rng.random((3, 20))
    objs = []
    W, H, _ = o.nmf_sparsity(X, 3, Winit=W0, Hinit=H0, sparsity=0, maxiter=200, trace=lambda it, W, H, of: objs.append(of))
    assert np.allclose(np.linalg.norm(W, axis=0), 1.0) and all(b <= a * (1 + 1e-10) for a, b in zip(objs, objs[1:]))
    _, Hs, _ = o.nmf_sparsity(X, 3, Winit=W0, Hinit=H0, sparsity=5.0, maxiter=200)
    assert Hs.sum() < H.sum()
    inf = {}
    o.nmf_sparsity(X, 3, Winit=W0, Hinit=H0, sparsity=0.1, maxiter=100000, tol=1e-6, info=inf)
    assert inf["stop_reason"] == "tol" and 1 < inf["iters"] < 100000


def test_execute_run_sparsity_composes_nmfsparsity_and_normalisation():
    """execute_run(...; method=:sparsity) reaches NMFsparsity through execute_singlerun_compute (NMFkExecute.jl:757-758): every
    restart equals nmf_sparsity followed by objvalue = normnan(X - W*H) (:791-792) and the H-row normalisation (:800-804), and
    the kw (cost_function, sparsity, lam) reach the solver."""
    rng = np.random.default_rng(12)
    X = np.asfortranarray(rng.random((25, 3)) @ rng.random((3, 12)) + 0.01)
    inits = [(rng.random((25, 3)), rng.random((3, 12))) for _ in range(4)]
    kw = dict(cost_function="kl", sparsity=0.2, lam=1e-8, maxiter=1000, tol=1e-6)
    det = {}
    Wa, Ha, phi, rob, aic = o.execute_run(X.copy(), 3, 4, inits=inits, method="sparsity", details=det, **kw)
    objs = []
    for i, (W0, H0) in enumerate(inits):
        inf = {}
        W, H, _ = o.nmf_sparsity(X.copy(), 3, Winit=W0, Hinit=H0, info=inf, **kw)
        objs.append(o.normnan(X - W @ H))
        total = H.sum(axis=1, keepdims=True)
        assert np.array_equal(det["WBig"][i], W * total.T) and np.array_equal(det["HBig"][i], H / total), i
        assert det["iters"][i] == inf["iters"] and det["stop_reasons"][i] == inf["stop_reason"], i
    assert np.array_equal(det["objvalue"], objs) and np.array_equal(det["idxsort"], np.argsort(objs, kind="stable"))
    assert set(det["stop_reasons"]) == {"tol"}  # tol reached: the keyword arrived
    _, _, objd = o.execute_singlerun_compute(X.copy(), 3, Winit=inits[0][0], Hinit=inits[0][1], maxiter=1000, tol=1e-6)
    assert objd != objs[0]  # method=:simple solves another problem
    with pytest.raises(ValueError):
        o.execute_singlerun_compute(X.copy(), 3, method="nmf", Winit=inits[0][0], Hinit=inits[0][1])
