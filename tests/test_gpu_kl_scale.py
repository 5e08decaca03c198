"""The KL tiled engine against the Float64 oracle (oracle/nmfk_oracle.py) at the batch sizes the benchmark solves.  The restart
count decides the slice count, the restart groups and the kernels that finish a run, so smaller batches at the same shapes run
other branches.  Inputs are built like bench.py: synth.mixture(..., seed=2015) and synth.philox_inits(2015, R, ...).

  test                                    shape, batch                      branches reached (nmfk.jl_b200/csrc/...)
  test_c3_as_benchmarked_vs_oracle        10000^2 f32 k=16 R=64, 10 it.     kl_tiled.cuh:763 slices() = 1 for both half-updates
                                                                            (16 groups of 4 restarts fill the grid): tc2_pass_kernel
                                                                            writes U itself, no combine (:965, :993: 3 + 3
                                                                            launches an iteration; R = 2 would take 4 + 4); tcgen05
                                                                            objective of the restart groups, tiled_check_kernel and
                                                                            its clamp (:1002-1055, n k < 2^18); restarts 0-3 (one
                                                                            group: both quotient groups, both accumulator slots), 33,
                                                                            62, 63 (the last group)
  test_c3_execute_run_decisions           the same, 20 it., normalize=1     capi.cu:1418 nmfk_execute_run -> finish_run (:1381):
                                                                            sort, clustersolutions, silhouettes, best restart with
                                                                            its signals permuted by the labels, phi and AIC
                                                                            (phi_aic, :1362) over 10^8 entries; two stop checks and
                                                                            tiled_finish_kernel's in-kernel normalisation
  test_c4_benchmark_batch_vs_oracle       100000 x 2000 f64 R=64, k=32, 5   DMMA pass (kl_tiled_dmma.cu) with an unsliced H-update:
                                                                            one launch over the whole 100 000-step reduction
                                                                            (2 + 2 launches an iteration)
  test_tall_clamp_and_normalisation       36000 x 120, k=8, n k >= 2^18,    kl_tiled.cuh:1021 tiled_clampW_kernel (:360; the
                                          R=6, f32 (tc2) and f64 (DMMA),    obj2 < tol early return, the grid-stride loop past its
                                          full stop rule, maxiter=40        first 36096 entries), :1083 the wide finish:
                                                                            tiled_finish_kernel leaves totals and wflag (:519-521),
                                                                            tiled_scaleW_kernel (:480) scales W; restarts that stop
                                                                            on the tolerance keep W entries below eps
  test_tall_resume_scales_once            the same, paused at 20            fin_flag cleared before the finish (:1084): a restart
                                                                            normalised in the first call is not scaled again
  test_c5_share_rowsharded_vs_oracle      500000 x 1000 f32 k=24 R=32,      row-sharded H-update (comm_init with one rank): tc_pass
                                          2 it.                             writes partials, dispatch_tiled_apply (:978-985) finishes
                                                                            (4 + 2 launches an iteration)

Tolerances are the north star's: 1e-4 relative for Float32 factors, 1e-9 for Float64, 2e-3 (Float32) and 1e-7 (Float64)
relative for objectives.  The oracle does most of the work: the restarts it solves are listed with each test.  It runs one
restart at a time (concurrent oracle runs in threads of one process gave wrong factors: its BLAS calls are not safe to
overlap)."""
import math

import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu
SEED = 2015
EPS64 = float(np.finfo(np.float64).eps)


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def ftol(dt):
    return 1e-9 if dt == np.float64 else 1e-4


def otol(dt):
    return 1e-7 if dt == np.float64 else 2e-3


def solve(ctx, k, W0, H0, **params):
    b = ctx.batch(k, W0.shape[0])
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(**params))
    out = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    return out


def launches_per_iteration(ctx, k, R, **params):
    """ctx.launches of a 2-iteration solve minus those of a 1-iteration one: the launches of one iteration without a stop
    check (kl_tiled.cuh:965 and :993 count them)."""
    def count(maxiter):
        b = ctx.batch(k, R)
        b.init_random(SEED)
        l0 = ctx.launches
        ctx.solve([b], nb.default_params(maxiter=maxiter, **params))
        b.close()
        return ctx.launches - l0
    return count(2) - count(1)


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


# ---- C3: 10000 x 10000 Float32, k = 16, 64 restarts ----------------------------------------------------------------------------
C3_N, C3_K, C3_R = 10000, 16, 64
C3_PROBE = (0, 1, 2, 3, 33, 62, 63)  # restarts 0 and 63 also take 20 iterations for the execute_run test


@pytest.fixture(scope="module")
def c3():
    """The C3 inputs and the oracle's state of the probed restarts after 10 iterations (W, H, the sum of squares of :125) and,
    for restarts 0 and 63, execute_singlerun_compute's result after 20 (normalised W, H, normnan objective)."""
    X = synth.mixture(C3_N, C3_N, 16, seed=SEED, dtype=np.float32)
    W0, H0 = synth.philox_inits(SEED, C3_R, C3_N, C3_K, C3_N, dtype=np.float32)
    X64 = np.asfortranarray(X.astype(np.float64))
    assert np.min(X64) > 0  # nothing for the oracle to substitute: it leaves X64 as it is

    def run(r):
        Wi, Hi = W0[r].astype(np.float64), H0[r].astype(np.float64)
        if r not in (0, C3_R - 1):
            W, H, ssq = o.nmf_multiplicative(X64, C3_K, Winit=Wi, Hinit=Hi, maxiter=10)
            return dict(at10=dict(W=W, H=H, ssq=ssq))
        at10 = {}

        def tr(it, W, H, obj):
            if it == 10:
                at10.update(W=W.copy(), H=H.copy())
        inf = {}
        W, H, phi = o.execute_singlerun_compute(X64, C3_K, Winit=Wi, Hinit=Hi, maxiter=20, trace=tr, info=inf)
        at10["ssq"] = float(np.sum((X64 - at10["W"] @ at10["H"]) ** 2))  # :125 after 10 iterations (X has no zeros)
        return dict(at10=at10, W=W, H=H, phi=phi, info=inf)
    ref = {r: run(r) for r in C3_PROBE}
    return dict(X=X, X64=X64, W0=W0, H0=H0, ref=ref)


def test_c3_as_benchmarked_vs_oracle(ctx, c3):
    """C3 with bench.py's batch (64 restarts, engine=2) for 10 iterations, normalize=0: every restart stops on maxiter; the
    probed restarts match the oracle in W, H and obj_ssq.  The launch count pins the configuration: one unsliced tc2
    half-update is 3 launches (column sums, V images, pass), a sliced one 4 (+ the combine)."""
    ctx.set_X(c3["X"])
    out = solve(ctx, C3_K, c3["W0"], c3["H0"], maxiter=10, engine=2, normalize=0)
    assert np.all(out["iters"] == 10) and np.all(out["stop_reason"] == 1), (out["iters"], out["stop_reason"])
    err = {}
    for r in C3_PROBE:
        ref = c3["ref"][r]["at10"]
        err[r] = (relerr(out["W"][r], ref["W"]), relerr(out["H"][r], ref["H"]), abs(out["obj_ssq"][r] - ref["ssq"]) / ref["ssq"])
        assert err[r][0] < 1e-4 and err[r][1] < 1e-4 and err[r][2] < 2e-3, (r, err[r])
    print("C3 R=64 largest relative differences: W %.2e, H %.2e, obj_ssq %.2e" % tuple(max(e[i] for e in err.values()) for i in range(3)))
    assert launches_per_iteration(ctx, C3_K, C3_R, engine=2, normalize=0) == 3 + 3


def test_c3_execute_run_decisions(ctx, c3):
    """execute_run's one-call form (nmfk_execute_run) at C3 with bench.py's inits, maxiter=20 and engine=2, against a batch solved
    with the same inputs and the oracle's post-processing of that batch's own 64 solutions: the best factors are the batch's
    restart order[0] with its signals permuted by the labels, bit for bit; labels are the oracle's; robustness, phi and AIC
    match the Float64 recomputation.  Restarts 0 and 63 (two stop checks, then normalisation) against
    execute_singlerun_compute."""
    X, W0, H0 = c3["X"], c3["W0"], c3["H0"]
    Wg, Hg, phi, rob, aic = nb.execute_run(X, C3_K, C3_R, inits=(W0, H0), maxiter=20, engine=2, ctx=ctx)
    ctx.set_X(X)
    b = ctx.batch(C3_K, C3_R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(maxiter=20, engine=2, normalize=1))
    sol = {key: np.array(v) for key, v in b.get().items()}
    cl = b.cluster()
    b.close()
    assert np.all(sol["iters"] == 20) and np.all(sol["stop_reason"] == 1)
    order = np.argsort(sol["obj_norm"].astype(np.float32), kind="stable")
    assert np.array_equal(cl["order"], order)
    ci = cl["labels"][:, 0] - 1
    best = order[0]
    assert np.array_equal(Wg, sol["W"][best][:, ci]) and np.array_equal(Hg, sol["H"][best][ci, :])
    # the oracle's clustering and silhouettes of the same 64 solutions, in Float64
    Hs = [sol["H"][i].astype(np.float64) for i in order]
    labels, _ = o.clustersolutions(Hs, False)
    assert np.array_equal(cl["labels"], labels)
    _, _, csil, _, _ = o.finalize([sol["W"][i].astype(np.float64) for i in order], Hs, labels, False)
    drob = abs(float(rob) - float(csil.min()))
    assert drob < 1e-6, (rob, csil.min())
    X64 = c3["X64"]
    phi64 = o.normnan(X64 - Wg.astype(np.float64) @ Hg.astype(np.float64))
    nobs = X64.size
    aic64 = 2 * (Wg.size + Hg.size) + nobs * math.log(phi64 / nobs)
    dphi = abs(float(phi) - phi64) / phi64
    assert dphi < 1e-6, (phi, phi64)
    assert abs(aic - aic64) <= nobs * 1e-6, (aic, aic64)  # d(AIC) = nobs d(phi) / phi
    err = []
    for r in (0, C3_R - 1):
        ref = c3["ref"][r]
        assert ref["info"]["iters"] == 20 and ref["info"]["stop_reason"] == "maxiter"
        err.append((relerr(sol["W"][r], ref["W"]), relerr(sol["H"][r], ref["H"]), abs(sol["obj_norm"][r] - ref["phi"]) / ref["phi"]))
        assert err[-1][0] < 1e-4 and err[-1][1] < 1e-4 and err[-1][2] < 2e-3, (r, err[-1])
        assert np.allclose(sol["H"][r].astype(np.float64).sum(axis=1), 1.0, rtol=0, atol=1e-5)
    print("C3 execute_run: robustness %.2e, phi %.2e, AIC %.3g (abs); restarts 0, 63: W %.2e, H %.2e, obj_norm %.2e"
          % ((drob, dphi, abs(aic - aic64)) + tuple(max(e[i] for e in err) for i in range(3))))


# ---- C4: 100000 x 2000 Float64, 64 restarts ------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4_X():
    X = synth.mixture(100000, 2000, 8, seed=SEED, dtype=np.float64)
    assert np.min(X) > 0
    return X


@pytest.mark.parametrize("k", [32, 5])
def test_c4_benchmark_batch_vs_oracle(ctx, c4_X, k):
    """C4 with a benchmark-sized batch (64 restarts, as each GPU of a 4-GPU run holds) on the DMMA pass: 2 iterations, restarts
    0, 31 and 63 against the oracle.  At 64 restarts the H-update (16 blocks of 128 columns x 64 restarts) fills the GPU without
    slicing its 100 000-step reduction: 2 + 2 launches an iteration (a sliced H-update would add its combine)."""
    X, R, niter = c4_X, 64, 2
    W0, H0 = synth.philox_inits(SEED, R, X.shape[0], k, X.shape[1])
    ctx.set_X(X)
    out = solve(ctx, k, W0, H0, maxiter=niter, engine=2, normalize=0)
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1)
    probe = [0, 31, 63]
    ref = {r: o.nmf_multiplicative(X, k, Winit=W0[r].copy(), Hinit=H0[r].copy(), maxiter=niter) for r in probe}
    err = []
    for r in probe:
        W, H, obj = ref[r]
        err.append((relerr(out["W"][r], W), relerr(out["H"][r], H), abs(out["obj_ssq"][r] - obj) / obj))
        assert err[-1][0] < 1e-9 and err[-1][1] < 1e-9 and err[-1][2] < 1e-7, (r, err[-1])
    print("C4 k=%d R=64 largest relative differences: W %.2e, H %.2e, obj_ssq %.2e" % ((k,) + tuple(max(e[i] for e in err) for i in range(3))))
    assert launches_per_iteration(ctx, k, R, engine=2, normalize=0) == 2 + 2


# ---- tall matrix: the whole-GPU clamp of the stop check and the whole-GPU W scaling of the normalisation ---------------------
# n k = 288 000 >= 2^18.  tiled_clampW_kernel runs 141 CTAs x 256 threads a restart, so its first pass covers entries 0 - 36095
# of the column-major W (column 0 and 96 rows of column 1) and the grid-stride loop the other 7 columns.  Rows TALL_ZERO of X are
# zero: lambda = 1e-32 after the preprocessing, and their W entries fall to ~1e-33 between two stop checks, so the clamp to
# eps(Float64) changes them (the oracle's trace shows it).  Restarts 1 and 4 start from blends of the mixture's own factors
# and reach a low objective early: tol between their objectives at iteration 10 and 20 (with every other restart above it
# at 40) stops exactly them on the tolerance at 20, where :75-78 leaves their W unclamped.  The Float32 data and initial
# factors are exactly representable in Float64, so one oracle run serves both types.
TALL_N, TALL_M, TALL_K, TALL_R = 36000, 120, 8, 6
TALL_ZERO = np.arange(37, TALL_N, 1999)
TALL_STOP = (1, 4)


@pytest.fixture(scope="module")
def tall():
    n, m, k, R = TALL_N, TALL_M, TALL_K, TALL_R
    X = synth.mixture(n, m, 8, seed=SEED, dtype=np.float32)
    X[TALL_ZERO, :] = 0
    rng = np.random.Generator(np.random.Philox(key=SEED))  # the factors synth.mixture multiplied
    Wt, Ht = rng.random((n, 8)), rng.random((8, m))
    W0, H0 = synth.philox_inits(SEED, R, n, k, m, dtype=np.float32)
    for r in TALL_STOP:
        W0[r] = (0.5 * W0[r] + 0.5 * Wt).astype(np.float32)
        H0[r] = (0.5 * H0[r] + 0.5 * Ht).astype(np.float32)
    X64 = np.asfortranarray(X.astype(np.float64))

    def run(r, tol=0.0, maxiter=40):
        objs, lamW = {}, {}

        def tr(it, W, H, obj):
            if obj is not None:
                objs[it] = obj
            if it in (9, 10):
                lamW[it] = W[TALL_ZERO].copy()
        inf = {}
        W, H, phi = o.execute_singlerun_compute(X64.copy(order="F"), k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64),
                                                maxiter=maxiter, tol=tol, trace=tr, info=inf)
        return dict(W=W, H=H, phi=phi, info=inf, objs=objs, lamW=lamW)
    free = {r: run(r) for r in range(R)}
    # tol: the geometric mean of the closest objectives on either side, at least 5 % from every objective that decides a stop
    below = max(free[r]["objs"][20] for r in TALL_STOP)
    above = min([free[r]["objs"][10] for r in TALL_STOP] + [free[r]["objs"][40] for r in range(R) if r not in TALL_STOP])
    tol = math.sqrt(below * above)
    assert below < tol / 1.05 and above > tol * 1.05, (below, tol, above)
    ref = dict(free)
    ref.update({r: run(r, tol) for r in TALL_STOP})
    return dict(X=X, W0=W0, H0=H0, tol=tol, ref=ref, free=free)


def _tall_inputs(tall, dt):
    return tall["X"].astype(dt), tall["W0"].astype(dt), tall["H0"].astype(dt)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_tall_clamp_and_normalisation(ctx, tall, dt):
    """Full stop rule (maxiter=40, tol from the oracle) and the default normalisation on a matrix with n k >= 2^18: Float32 on
    the tc2 pass, Float64 on the DMMA pass.  Iteration counts and stop reasons equal the oracle's; W and H after the
    normalisation match per restart, and so do the W rows of the zeroed X rows on their own scale: the clamp to eps(Float64)
    in every column for the restarts that go on, none for the two that stop on the tolerance at iteration 20."""
    ref, R = tall["ref"], TALL_R
    for r in range(R):  # the oracle's trace: the lambda rows are below eps in every column before the first check, eps after it
        assert np.all(tall["free"][r]["lamW"][9].max(axis=0) < EPS64), r
        assert np.all(tall["free"][r]["lamW"][10] == EPS64), r
    X, W0, H0 = _tall_inputs(tall, dt)
    ctx.set_X(X)
    out = solve(ctx, TALL_K, W0, H0, maxiter=40, tol=tall["tol"], engine=2)
    reason = {"tol": 2, "maxiter": 1}
    err = []
    for r in range(R):
        inf = ref[r]["info"]
        assert out["iters"][r] == inf["iters"] and out["stop_reason"][r] == reason[inf["stop_reason"]], (r, out["iters"][r], inf)
        assert (inf["iters"], inf["stop_reason"]) == ((20, "tol") if r in TALL_STOP else (40, "maxiter")), (r, inf)
        W, H = out["W"][r], out["H"][r]
        e = (relerr(W, ref[r]["W"]), relerr(H, ref[r]["H"]), relerr(W[TALL_ZERO], ref[r]["W"][TALL_ZERO]),
             abs(out["obj_norm"][r] - ref[r]["phi"]) / ref[r]["phi"])
        err.append(e)
        assert e[0] < ftol(dt) and e[1] < ftol(dt) and e[2] < ftol(dt) and e[3] < otol(dt), (r, e)
        assert np.allclose(H.astype(np.float64).sum(axis=1), 1.0, rtol=0, atol=1e-5 if dt == np.float32 else 1e-12), r
        if r in TALL_STOP:  # stopped on the tolerance before the clamp of :100: W * total still holds entries below eps
            assert np.max(W[TALL_ZERO]) < EPS64 and np.max(ref[r]["W"][TALL_ZERO]) < EPS64, r
    print("tall %s: largest relative differences W %.2e, H %.2e, lambda rows of W %.2e, obj_norm %.2e"
          % ((np.dtype(dt).name,) + tuple(max(e[i] for e in err) for i in range(4))))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_tall_resume_scales_once(ctx, tall, dt):
    """The batch of test_tall_clamp_and_normalisation paused with iter_limit=20 and resumed: restarts 1 and 4 stop on the
    tolerance and are normalised in the first call, the others in the second; the result equals the continuous run bit for
    bit, so the second call's whole-GPU W scaling leaves the restarts finished in the first one alone."""
    X, W0, H0 = _tall_inputs(tall, dt)
    ctx.set_X(X)
    p = dict(maxiter=40, tol=tall["tol"], engine=2)
    cont = solve(ctx, TALL_K, W0, H0, **p)
    b = ctx.batch(TALL_K, TALL_R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(iter_limit=20, **p))
    mid = b.get(factors=False)
    assert [int(mid["stop_reason"][r]) for r in range(TALL_R)] == [2 if r in TALL_STOP else 0 for r in range(TALL_R)], mid["stop_reason"]
    ctx.solve([b], nb.default_params(**p))
    res = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    for key in ("iters", "stop_reason", "obj_norm", "W", "H"):
        assert np.array_equal(res[key], cont[key]), key


# ---- one rank's share of C5 through the row-sharded path ---------------------------------------------------------------------
def test_c5_share_rowsharded_vs_oracle():
    """500000 x 1000 Float32, k = 24, 32 restarts (the C5 batch) on a row-sharded context of one rank: tc_pass_kernel leaves the
    H-update numerators as partials and the apply kernel finishes them after the (single-rank) all-reduce, 4 + 2 launches an
    iteration.  2 iterations; restarts 0, 15 and 31 against the oracle."""
    n, m, k, R, niter = 500000, 1000, 24, 32, 2
    X = synth.mixture(n, m, 24, seed=SEED, dtype=np.float32)
    W0, H0 = synth.philox_inits(SEED, R, n, k, m, dtype=np.float32)
    with nb.Context() as c:
        c.comm_init(1, 0, None, 0, n)
        c.set_X(X)
        out = solve(c, k, W0, H0, maxiter=niter, engine=2, normalize=0)
        per_it = launches_per_iteration(c, k, R, engine=2, normalize=0)
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1)
    X64 = np.asfortranarray(X.astype(np.float64))
    del X
    assert np.min(X64) > 0
    probe = [0, 15, 31]
    ref = {r: o.nmf_multiplicative(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=niter) for r in probe}
    err = []
    for r in probe:
        W, H, obj = ref[r]
        err.append((relerr(out["W"][r], W), relerr(out["H"][r], H), abs(out["obj_ssq"][r] - obj) / obj))
        assert err[-1][0] < 1e-4 and err[-1][1] < 1e-4 and err[-1][2] < 2e-3, (r, err[-1])
    print("C5 share R=32 largest relative differences: W %.2e, H %.2e, obj_ssq %.2e" % tuple(max(e[i] for e in err) for i in range(3)))
    assert per_it == 4 + 2, per_it
