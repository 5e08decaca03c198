"""Variant FRO (method=:nmf, algorithm=:multdiv -> NMF.MultUpdate(obj=:mse); the update BASELINE.json's north star writes out) on
the GPU against the oracle's restatement of NMF.jl (oracle/nmfk_oracle.py::nmf_multupdate_mse):
the stacked-restart GEMM alone (tcgen05 3xTF32 / DMMA) against NumPy, then per-iteration factors, the stop rule, and execute
with method="nmf".  Tolerances: 1e-9 relative for Float64, 1e-4 for Float32 (north star)."""
import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


@pytest.mark.parametrize("M,N,K", [(128, 256, 32), (128, 256, 256), (256, 512, 1024), (1024, 1000, 2000), (48, 100, 36), (300, 260, 4100)])
def test_stacked_gemm_f32_3xtf32(ctx, M, N, K):
    """C = A B^T on tcgen05 with the 3-term TF32 split: FP32-level accuracy (plain TF32 would be ~1e-3), edge tiles in M, N, K."""
    rng = np.random.default_rng(M + N + K)
    A = rng.random((M, K), dtype=np.float32)
    B = rng.random((N, K), dtype=np.float32)
    C, ms = ctx.gemm_nt(A, B)
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    assert relerr(C, ref) < 1e-5, relerr(C, ref)  # round-toward-zero chains of 96 instructions: ~ -5e-6
    # exactly representable inputs (TF32-exact, small K): the product is exact
    Ai = rng.integers(0, 64, (M, K)).astype(np.float32)
    Bi = rng.integers(0, 64, (N, K)).astype(np.float32)
    Ci, _ = ctx.gemm_nt(Ai[:, :32].copy(), Bi[:, :32].copy())
    assert np.array_equal(Ci.astype(np.float64), Ai[:, :32].astype(np.float64) @ Bi[:, :32].astype(np.float64).T)


@pytest.mark.parametrize("M,N,K", [(128, 128, 16), (256, 384, 1000), (100, 77, 333), (512, 2000, 1001)])
def test_stacked_gemm_f64_dmma(ctx, M, N, K):
    rng = np.random.default_rng(M * 3 + N + K)
    A = rng.random((M, K))
    B = rng.random((N, K))
    C, ms = ctx.gemm_nt(A, B)
    assert relerr(C, A @ B.T) < 1e-13


def _trace_fro(ctx, X, k, W0, H0, niter, dt):
    ctx.set_X(X)
    b = ctx.batch(k, W0.shape[0])
    b.set_init(W0, H0)
    outs = []
    for t in range(1, niter + 1):
        ctx.solve([b], nb.default_params(variant=1, maxiter=10 ** 6, iter_limit=t, normalize=0))
        g = b.get()
        outs.append((g["W"].copy(), g["H"].copy()))
    b.close()
    return outs


@pytest.mark.parametrize("n,m,k,R,niter,dt", [(512, 256, 8, 3, 12, np.float32), (1000, 200, 10, 2, 10, np.float64),
                                              (300, 64, 13, 2, 8, np.float64), (2048, 1024, 16, 5, 8, np.float32),
                                              (128, 64, 1, 2, 6, np.float32), (260, 132, 3, 2, 10, np.float32)])
def test_fro_per_iteration_vs_oracle(ctx, n, m, k, R, niter, dt):
    """Per-iteration W, H of the stacked FRO solve against the Float64 oracle from the same initial factors."""
    X = synth.mixture(n, m, 3, seed=17, dtype=dt)
    W0, H0 = synth.philox_inits(23, R, n, k, m, dtype=dt)
    outs = _trace_fro(ctx, X, k, W0, H0, niter, dt)
    tol = 1e-9 if dt == np.float64 else 1e-4
    delta = float(np.sqrt(np.finfo(dt).eps))
    X64 = X.astype(np.float64)
    for r in range(R):
        ref = []
        o.nmf_multupdate_mse(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=niter, tol=0.0, delta=delta,
                             trace=lambda it, W, H: ref.append((W.copy(), H.copy())))
        for t in range(niter):
            assert relerr(outs[t][0][r], ref[t][0]) < tol, ("W", r, t, relerr(outs[t][0][r], ref[t][0]))
            assert relerr(outs[t][1][r], ref[t][1]) < tol, ("H", r, t, relerr(outs[t][1][r], ref[t][1]))


def test_fro_stop_rule_and_execute(ctx):
    """NMF.jl stop_condition (relative change of every column of W / row of H below tol) with a loose tol: same iteration count as
    the oracle; then execute(X, ks, nNMF; method=:nmf, algorithm=:multdiv): objective = normnan(X - W*H), rows of H sum to one,
    kopt and robustness against the oracle's execute_run fed with the same solver."""
    X = synth.mixture(400, 120, 3, seed=5)
    k, R = 3, 4
    W0, H0 = synth.philox_inits(9, R, 400, k, 120)
    ctx.set_X(X)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(variant=1, maxiter=5000, tol=1e-4))
    g = b.get()
    b.close()
    for r in range(R):
        inf = {}
        W, H, obj = o.execute_singlerun_nmf(X.copy(), k, Winit=W0[r].copy(), Hinit=H0[r].copy(), maxiter=5000, tol=1e-4, info=inf)
        assert g["iters"][r] == inf["iters"] and g["stop_reason"][r] == 2, (r, g["iters"][r], inf)
        assert relerr(g["W"][r], W) < 1e-7 and relerr(g["H"][r], H) < 1e-7 and abs(g["obj_norm"][r] - obj) <= 1e-7 * obj + 1e-12
        assert np.allclose(g["H"][r].sum(axis=1), 1.0, atol=1e-12)
    # through the reference-shaped entry with the reference's keywords
    Wg, Hg, fg, rg, ag = nb.execute_run(X, k, R, inits=(W0, H0), method="nmf", algorithm="multdiv", maxiter=300, ctx=ctx)
    sols = [o.execute_singlerun_nmf(X.copy(), k, Winit=W0[r].copy(), Hinit=H0[r].copy(), maxiter=300) for r in range(R)]
    best = int(np.argmin([s[2] for s in sols]))
    assert abs(fg - sols[best][2]) <= 1e-7 * sols[best][2]
    labels, _ = o.clustersolutions([sols[i][1] for i in np.argsort([s[2] for s in sols], kind="stable")], False)
    _, _, csil, _, _ = o.finalize([s[0] for s in sols], [sols[i][1] for i in np.argsort([s[2] for s in sols], kind="stable")], labels, False)
    assert abs(rg - float(csil.min())) < 1e-7
    with pytest.raises(nb.NMFkError):
        nb.execute_run(X, k, R, method="nmf", algorithm="alspgrad", ctx=ctx)


# ---- the stacked solve at the shapes the benchmark and larger restart counts reach -------------------------------------------
# The launch choices of solve_fro_t and fro_gemm_slices depend on shape (below for 148 SMs, worked out from the code):
#   case                      R*k  M tiles  cluster  split-K H/W  Gram SW/SH  apply KMAX  restarts across a 128-row M tile
#   4100 x 1204 k=12 R=23 f32  276  3        2        7 / 2        2 / 1       16          10 (tiles 0|1), 21 (1|2: cluster pair)
#   1204 x 4100 k=20 R=13 f32  260  3        2        2 / 7        1 / 2       32          6, 12
#   8192 x 640  k=24 R=11 f32  264  3        2        12 / 1       4 / 1       32          5, 10
#   1028 x 2052 k=32 R=5  f32  160  2        2        2 / 4        1 / 1       32          -
#   2049 x 1027 k=20 R=9  f64  180  2        -        DMMA, odd n and m: fro_gemm_f64_kernel<false> (unaligned loads)    6
# What runs where:
#   1. fro_gemm_kernel<2> (cluster multicast) inside a solve, split-K partials summed by fro_apply_kernel's NS loop:
#      every f32 case above, test_c3_variant_fro_vs_oracle (tests/test_gpu_configs.py, 8 tiles, 6 / 6 slices) and the
#      slice-count test (NMFK_FRO_SLICES = 1, default, 5; NMFK_FRO_CLUSTER = 1)
#   2. restarts across an M tile or a cluster pair: the 4100 / 1204 / 8192 / 2049 cases, the stop-rule tests
#   3. sliced Gram (SW, SH > 1): 4100 x 1204 (SW 2), 1204 x 4100 (SH 2), 8192 x 640 (SW 4), C3 (4 / 4)
#   4. k = 17 ... 32 (fro_apply_kernel<T, 32>, Gram pairs >= 256): k = 20, 24, 32 (pairs up to 1023 fill acc[0..3])
#   5. Float32 NMF.jl stop rule with frozen restarts in a running 3-tile stack: test_fro_float32_stop_rule_frozen_restarts
#   6. Float32 post-run objective (tcgen05, obj_sel = obj_restore = 1) and normalisation: test_fro_float32_objective_and_normalisation
#   7. Float64 with odd n, m (unaligned DMMA GEMM): 2049 x 1027, test_fro_float64_stop_rule_multi_tile_odd_n
#   8. pause (iter_limit) and resume: test_fro_resume_equals_continuous
MULTI_TILE = [(4100, 1204, 12, 23, np.float32), (1204, 4100, 20, 13, np.float32), (8192, 640, 24, 11, np.float32),
              (1028, 2052, 32, 5, np.float32), (2049, 1027, 20, 9, np.float64)]


def _probe_restarts(R, k):
    """Restarts whose k rows of the [R*k]-row stack lie in the first 128-row M tile, in the second (the second CTA of a cluster
    pair), in the last (ragged) tile, and every restart that crosses a tile boundary."""
    tiles = [(r * k // 128, ((r + 1) * k - 1) // 128) for r in range(R)]
    rs = {0, R - 1} | {r for r, (a, b) in enumerate(tiles) if a != b}
    rs |= {next(r for r, (a, b) in enumerate(tiles) if a == b == 1)} if any(a == b == 1 for a, b in tiles) else set()
    return sorted(rs)


def _oracle(X64, k, W0, H0, niter, dt, tol=0.0, trace=None, info=None):
    return o.nmf_multupdate_mse(X64, k, Winit=W0.astype(np.float64), Hinit=H0.astype(np.float64), maxiter=niter, tol=tol,
                                delta=float(np.sqrt(np.finfo(dt).eps)), trace=trace, info=info)


def _fro_solve(ctx, k, W0, H0, **params):
    b = ctx.batch(k, W0.shape[0])
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(variant=1, **params))
    g = b.get()
    b.close()
    return {key: np.array(v) for key, v in g.items()}


def _assert_no_timeout(capfd):
    err = capfd.readouterr().err
    assert "barrier time-out" not in err, err[-2000:]


def _fixed_iterations_check(out, X, k, W0, H0, niter, dt, restarts):
    tol = 1e-9 if dt == np.float64 else 1e-4
    X64 = X.astype(np.float64)
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1), (out["iters"], out["stop_reason"])
    for r in restarts:
        W, H, _ = _oracle(X64, k, W0[r], H0[r], niter, dt)
        eW, eH = relerr(out["W"][r], W), relerr(out["H"][r], H)
        assert eW < tol and eH < tol, (r, eW, eH)


@pytest.mark.parametrize("n,m,k,R,dt", MULTI_TILE)
def test_fro_multi_tile_stack_vs_oracle(ctx, capfd, n, m, k, R, dt):
    """One continuous solve (maxiter = 4, normalize = 0) of a stack of several 128-row M tiles against the Float64 oracle:
    restarts of the first, second and last tile and every restart across a tile boundary (the restarts of a stack are
    independent: each reads only its own rows of the stacked GEMM)."""
    X = synth.mixture(n, m, 5, seed=2017, dtype=dt)
    W0, H0 = synth.philox_inits(29, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    out = _fro_solve(ctx, k, W0, H0, maxiter=4, normalize=0)
    _fixed_iterations_check(out, X, k, W0, H0, 4, dt, _probe_restarts(R, k))
    _assert_no_timeout(capfd)


def test_fro_split_k_and_cluster_choice_do_not_change_results(ctx, capfd, monkeypatch, tmp_path):
    """The split-K slice count (NMFK_FRO_SLICES: 1, the default 7 / 2, and 5, which divides neither 129 nor 38 K-blocks) and the
    cluster multicast (NMFK_FRO_CLUSTER=1, read once per process: in a child process) only reorder the sums of the stacked
    GEMM: every run matches the oracle, and all agree within 2e-5."""
    import os
    import subprocess
    import sys
    n, m, k, R, dt, niter = 4100, 1204, 12, 23, np.float32, 4
    X = synth.mixture(n, m, 5, seed=2017, dtype=dt)
    W0, H0 = synth.philox_inits(29, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    runs = {}
    for slices in ("1", None, "5"):
        if slices is None:
            monkeypatch.delenv("NMFK_FRO_SLICES", raising=False)
        else:
            monkeypatch.setenv("NMFK_FRO_SLICES", slices)
        runs[slices] = _fro_solve(ctx, k, W0, H0, maxiter=niter, normalize=0)
        _fixed_iterations_check(runs[slices], X, k, W0, H0, niter, dt, _probe_restarts(R, k))
    monkeypatch.delenv("NMFK_FRO_SLICES", raising=False)
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    np.savez(tmp_path / "in.npz", X=X, W0=W0, H0=H0)
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import nmfk_b200 as nb\n"
        "d = np.load(%r)\n"
        "with nb.Context(0) as ctx:\n"
        "    ctx.set_X(d['X'])\n"
        "    b = ctx.batch(%d, %d); b.set_init(d['W0'], d['H0'])\n"
        "    ctx.solve([b], nb.default_params(variant=1, maxiter=%d, normalize=0))\n"
        "    g = b.get(); np.savez(%r, W=g['W'], H=g['H'], iters=g['iters'])\n"
    ) % (os.path.join(ROOT, "nmfk.jl_b200", "python"), ROOT, str(tmp_path / "in.npz"), k, R, niter, str(tmp_path / "c1.npz"))
    env = {key: v for key, v in os.environ.items() if key != "NMFK_FRO_SLICES"}
    env["NMFK_FRO_CLUSTER"] = "1"
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "barrier time-out" not in r.stderr, r.stderr[-2000:]
    c1 = np.load(tmp_path / "c1.npz")
    runs["cluster1"] = {"W": c1["W"], "H": c1["H"], "iters": c1["iters"]}
    _fixed_iterations_check(dict(runs["cluster1"], stop_reason=np.ones(R)), X, k, W0, H0, niter, dt, _probe_restarts(R, k))
    for key, g in runs.items():
        assert relerr(g["W"], runs[None]["W"]) < 2e-5 and relerr(g["H"], runs[None]["H"]) < 2e-5, key
    _assert_no_timeout(capfd)


def test_fro_resume_equals_continuous(ctx, capfd):
    """t solves of one iteration each (iter_limit pauses the run; the next call re-stacks H and rebuilds the lo images of the
    3-term split from the API copies, with the formulas the apply kernel uses) against one t-iteration solve: bit-identical."""
    n, m, k, R, dt, niter = 4100, 1204, 12, 23, np.float32, 4
    X = synth.mixture(n, m, 5, seed=2017, dtype=dt)
    W0, H0 = synth.philox_inits(31, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    cont = _fro_solve(ctx, k, W0, H0, maxiter=niter, normalize=0)
    b = ctx.batch(k, R)
    b.set_init(W0, H0)
    for t in range(1, niter + 1):
        ctx.solve([b], nb.default_params(variant=1, maxiter=10 ** 6, iter_limit=t, normalize=0))
    g = b.get()
    b.close()
    assert np.array_equal(g["iters"], cont["iters"])
    assert np.array_equal(g["W"], cont["W"]) and np.array_equal(g["H"], cont["H"])
    _assert_no_timeout(capfd)


def test_fro_batch_composition(ctx, capfd):
    """A restart solved alone and inside a batch: Float64 bit-identical (the DMMA accumulation order of an element does not
    depend on M; Gram and apply run per restart), Float32 within 2e-5 (the split-K slice count depends on R*k).  Then three
    batches of different k in one solve call against three separate calls, bit for bit (no scratch reused stale)."""
    for n, m, k, R, r, dt in ((2049, 1027, 20, 9, 6, np.float64), (4100, 1204, 12, 23, 10, np.float32)):
        X = synth.mixture(n, m, 5, seed=2017, dtype=dt)
        W0, H0 = synth.philox_inits(29, R, n, k, m, dtype=dt)
        ctx.set_X(X)
        batch = _fro_solve(ctx, k, W0, H0, maxiter=4, normalize=0)
        alone = _fro_solve(ctx, k, W0[r:r + 1], H0[r:r + 1], maxiter=4, normalize=0)
        if dt == np.float64:
            assert np.array_equal(alone["W"][0], batch["W"][r]) and np.array_equal(alone["H"][0], batch["H"][r])
        else:
            assert relerr(alone["W"][0], batch["W"][r]) < 2e-5 and relerr(alone["H"][0], batch["H"][r]) < 2e-5
    n, m = 1028, 2052
    X = synth.mixture(n, m, 5, seed=2019, dtype=np.float32)
    ctx.set_X(X)
    specs = [(5, 30), (12, 11), (20, 7)]
    inits = [synth.philox_inits(40 + k, R, n, k, m, dtype=np.float32) for k, R in specs]
    p = nb.default_params(variant=1, maxiter=5, normalize=0)
    bs = []
    for (k, R), (W0, H0) in zip(specs, inits):
        b = ctx.batch(k, R)
        b.set_init(W0, H0)
        bs.append(b)
    ctx.solve(bs, p)
    together = [b.get() for b in bs]
    for b in bs:
        b.close()
    for (k, R), (W0, H0), g in zip(specs, inits, together):
        sep = _fro_solve(ctx, k, W0, H0, maxiter=5, normalize=0)
        assert np.array_equal(g["W"], sep["W"]) and np.array_equal(g["H"], sep["H"]), k
        assert np.array_equal(g["iters"], sep["iters"]) and np.array_equal(g["obj_norm"], sep["obj_norm"]), k
    _assert_no_timeout(capfd)


def _stop_criterion(trace, W0, H0):
    """NMF.jl stop_condition of every iteration of an oracle trace: c(i) = max over columns of W and rows of H of
    sqrt(sum((new - old)^2)) / sqrt(sum((new + old)^2)); the run stops at the first i with c(i) <= tol."""
    c, pW, pH = [], W0, H0
    for W, H in trace:
        cw = np.sqrt(((W - pW) ** 2).sum(axis=0)) / np.sqrt(((W + pW) ** 2).sum(axis=0))
        ch = np.sqrt(((H - pH) ** 2).sum(axis=1)) / np.sqrt(((H + pH) ** 2).sum(axis=1))
        c.append(max(cw.max(), ch.max()))
        pW, pH = W, H
    return np.array(c)


# bound on the relative difference between the Float32 device factors at their stop iteration and the Float64 oracle at the
# same iteration in test_fro_float32_stop_rule_frozen_restarts: 5 x the 4.1e-5 measured on a B200 (1000 W power limit)
F32_STOP_DRIFT = 2e-4


def test_fro_float32_stop_rule_frozen_restarts(ctx, capfd):
    """Float32 NMF.jl stop rule in a 3-tile stack (R*k = 260, k = 20, tol = 3e-3): restarts stop at different iterations and
    then sit frozen while the rest of the stack keeps running through the same GEMMs.  Every restart stops by the rule
    (stop_reason 2); the stop iteration t satisfies the oracle's criterion, c(t) < tol (1 + eps) and c(t - 1) >= tol (1 - eps)
    with eps = 5 % for the Float32 / Float64 trajectory difference; the factors match the oracle at iteration t within
    F32_STOP_DRIFT (measured on a B200: stop iterations 62 - 69, the same as the oracle's, and a largest relative difference
    of 4.1e-5 after them)."""
    n, m, k, R, dt, tol = 1204, 404, 20, 13, np.float32, 3e-3
    X = synth.mixture(n, m, 4, seed=7, dtype=dt)
    W0, H0 = synth.philox_inits(11, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    out = _fro_solve(ctx, k, W0, H0, maxiter=1000, tol=tol, normalize=0)
    assert np.all(out["stop_reason"] == 2), out["stop_reason"]
    assert len(set(out["iters"].tolist())) >= 3, out["iters"]
    X64 = X.astype(np.float64)
    eps = 0.05
    drift = []
    for r in range(R):
        t = int(out["iters"][r])
        tr = []
        _oracle(X64, k, W0[r], H0[r], t, dt, trace=lambda it, W, H: tr.append((W.copy(), H.copy())))
        c = _stop_criterion(tr, W0[r].astype(np.float64), H0[r].astype(np.float64))
        assert c[t - 1] < tol * (1 + eps) and c[t - 2] >= tol * (1 - eps), (r, t, c[t - 3:t] / tol)
        drift.append(max(relerr(out["W"][r], tr[t - 1][0]), relerr(out["H"][r], tr[t - 1][1])))
    assert max(drift) < F32_STOP_DRIFT, drift
    _assert_no_timeout(capfd)


def test_fro_float64_stop_rule_multi_tile_odd_n(ctx, capfd):
    """Float64 stop rule at R*k = 150 (2 M tiles, restart 12 across them) with odd n: the same iteration count as the oracle
    for every restart (its criterion is at least 0.16 % away from tol at the deciding iterations), factors within 1e-9."""
    n, m, k, R, dt, tol = 1001, 300, 10, 15, np.float64, 1e-3
    X = synth.mixture(n, m, 3, seed=5, dtype=dt)
    W0, H0 = synth.philox_inits(9, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    out = _fro_solve(ctx, k, W0, H0, maxiter=1000, tol=tol, normalize=0)
    err = []
    for r in range(R):
        inf = {}
        W, H, _ = _oracle(X, k, W0[r], H0[r], 1000, dt, tol=tol, info=inf)
        assert out["iters"][r] == inf["iters"] and out["stop_reason"][r] == 2, (r, out["iters"][r], inf)
        err.append(max(relerr(out["W"][r], W), relerr(out["H"][r], H)))
    assert max(err) < 1e-9, err  # 1.2e-14 measured on a B200
    _assert_no_timeout(capfd)


@pytest.mark.parametrize("n,m,k,R", [(1156, 840, 12, 13), (2052, 1028, 20, 9), (516, 260, 3, 4)])
def test_fro_float32_objective_and_normalisation(ctx, capfd, n, m, k, R):
    """Float32 post-run objective (the tcgen05 objective kernel, obj_sel = obj_restore = 1; n = 1156 and 516 are not multiples of
    128) and normalisation: obj_norm = ||X - W H||_F in Float64 from the returned factors within 1e-5 ||W H||_F (the 3xTF32
    product error; W, H >= 0), obj_ssq = obj_norm^2 (weight 1), obj_norm against the oracle's objvalue, rows of H sum to 1."""
    dt, niter = np.float32, 5
    X = synth.mixture(n, m, 4, seed=13, dtype=dt)
    W0, H0 = synth.philox_inits(17, R, n, k, m, dtype=dt)
    ctx.set_X(X)
    out = _fro_solve(ctx, k, W0, H0, maxiter=niter)
    X64 = X.astype(np.float64)
    for r in range(R):
        WH = out["W"][r].astype(np.float64) @ out["H"][r].astype(np.float64)
        nWH = np.linalg.norm(WH)
        ref = np.linalg.norm(X64 - WH)
        assert abs(out["obj_norm"][r] - ref) <= 1e-5 * nWH, (r, out["obj_norm"][r], ref, nWH)
        assert abs(out["obj_ssq"][r] - out["obj_norm"][r] ** 2) <= 1e-12 * out["obj_ssq"][r], r
        _, _, objo = o.execute_singlerun_nmf(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=niter,
                                             delta=float(np.sqrt(np.finfo(dt).eps)))
        assert abs(out["obj_norm"][r] - objo) <= 1e-4 * nWH, (r, out["obj_norm"][r], objo, nWH)
        assert np.allclose(out["H"][r].astype(np.float64).sum(axis=1), 1.0, rtol=0, atol=1e-5), r
    _assert_no_timeout(capfd)


def test_fro_refusals(ctx):
    """Variant FRO refuses, with NMFK_E_UNSUPPORTED: Float32 X with n or m not a multiple of 4 (TMA strides), k = 33, NaN in X."""
    unsupported = -6
    p = nb.default_params(variant=1, maxiter=2)
    for n, m in ((402, 120), (400, 122)):
        ctx.set_X(synth.mixture(n, m, 3, seed=5, dtype=np.float32))
        b = ctx.batch(3, 2)
        b.init_random(1)
        with pytest.raises(nb.NMFkError) as e:
            ctx.solve([b], p)
        b.close()
        assert e.value.status == unsupported, (n, m, e.value)
    for dt in (np.float32, np.float64):
        ctx.set_X(synth.mixture(400, 120, 3, seed=5, dtype=dt))
        b = ctx.batch(33, 1)
        b.init_random(1)
        with pytest.raises(nb.NMFkError) as e:
            ctx.solve([b], p)
        b.close()
        assert e.value.status == unsupported, (dt, e.value)
        X = synth.mixture(400, 120, 3, seed=5, dtype=dt)
        X[7, 11] = np.nan
        ctx.set_X(X)
        b = ctx.batch(3, 2)
        b.init_random(1)
        with pytest.raises(nb.NMFkError) as e:
            ctx.solve([b], p)
        b.close()
        assert e.value.status == unsupported, (dt, e.value)
