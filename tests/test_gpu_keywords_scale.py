"""The keywords of NMFmultiplicative / execute (Wfixed, Hfixed, weight, normalizevector) and missing entries on the KL tiled
engine against the Float64 oracle (oracle/nmfk_oracle.py), at shapes and batches where the engine picks its tensor-core
passes (or, with NaN, its sliced scalar pass).  At the sizes of tests/test_gpu_keywords.py the same keywords run the resident
engine or a one-block scalar pass.  Inputs are built like bench.py: synth.mixture(..., seed=2015) and
synth.philox_inits(2015, R, ...).

  test                                   shape, batch                        branches reached (nmfk.jl_b200/csrc/...)
  test_fixed_factor_on_tensor_passes     12000 x 1000 f32 k=16 R=16 Hfixed   kl_tiled.cuh:959 H-update skipped; tc2 W-update from
                                                                             V images of the fixed H, unsliced (3 launches an it.)
                                         20000 x 512 f32 k=24 R=8 Wfixed     gen-1 tc_pass H-update sliced 30 ways + combine (3)
                                         20000 x 512 f32 k=24 R=8 Hfixed     gen-1 tc_pass W-update, unsliced (2)
                                         40000 x 600 f64 k=8 R=8 Wfixed      DMMA H-update sliced 14 ways + combine (3)
                                         40000 x 600 f64 k=8 R=8 Hfixed      DMMA W-update, unsliced (2)
                                         all: 10 it., fixed entries 0 and    Wfixed with n k >= 2^18: wide_clamp off (:1021), so
                                         1e-300                              tiled_check_kernel clamps W in one CTA (:425); H is
                                                                             clamped there always (:430): the fixed factor comes
                                                                             back as max(F, eps) exactly, like the oracle's :202-203
  test_caller_patterns_draw_the_free_factor  24000 x 400 f64 k=16 R=8        execute_k(seed, Hinit, Hfixed) / execute_run(seed,
                                         and its transpose, 10 it.           Winit, Wfixed): preprocess.cu:123-150 draws only the
                                                                             free factor from the start of each restart's Philox
                                                                             stream (3 072 000 numbers, 5 x the grid's threads: the
                                                                             grid-stride loop); DMMA half-update alone (2); no
                                                                             normalisation or signal reordering (api.py:486, 557)
  test_weights_with_the_stop_rule        3000 x 1000 R=16, 1 % zeros,        scalar weight: the weighted objective of the tc pass
                                         f32 k=8 (tc2, 4 + 3 launches),      (kl_tiled_tc.cu:387) and of the DMMA pass
                                         f32 k=20 (gen-1, 3 + 2),            (kl_tiled_dmma.cu:208) in every stop check and the final
                                         f64 k=8 (DMMA, 3 + 2);              sum; row / column / matrix weights: wobj (:783) sends the
                                         maxiter 40, tol / tolOF from the    checks and the final sum to tiled_objective_kernel
                                         oracle trace, maxbaditers=2,        (weight_at, nmfk_internal.h:47) next to the tensor-core
                                         maxreattempts=1                     passes over 24 row blocks and 16 restarts
  test_normalizevector_batch             2500 x 1012 R=8, 20 it., normalize  set_X's Xn = X ./ nv feeds the tc2 / gen-1 / DMMA passes;
                                         =1: f32 k=8, f32 k=20, f64 k=8,     capi.cu:763 finish_normalizevector for every restart:
                                         f64 k=8 with a row weight           W .*= nv, residual() against the caller's X (with the
                                                                             array weight), renormalize_kernel (preprocess.cu:220)
  test_normalizevector_clusterW_tall     36004 x 124 k=8 R=1, f32 and f64    execute_singlerun(clusterWmatrix=true): normalize = 2
                                                                             in renormalize_kernel; tiled_clampW_kernel (n k >= 2^18)
  test_normalizevector_resume            2500 x 1012 k=8 R=8, f32 and f64,   restarts 2 and 5 stop on tol at 10 and are scaled in the
                                         iter_limit=10, then maxiter=20      first call; done = 2 keeps the second call off them
  test_missing_entries_at_scale          8192 x 1024 k=12 R=8, 5 % NaN,      HASNAN scalar pass, both half-updates sliced (21 x 4 f32,
                                         1 % zeros, f32 and f64              21 x 4 f64) + combines + tiled_impute_kernel: 7 launches an
                                                                             iteration (R = 1: 32 / 64 x 4 slices); the per-restart
                                                                             store r n m (:71, :332); the final objective without the
                                                                             NaN entries; a resume at 10 rebuilds ximp (:923-929) and
                                                                             reads it (first_iter only at iteration 1, :958)

Tolerances are the north star's: 1e-4 relative for Float32 factors, 1e-9 for Float64, 2e-3 (Float32) and 1e-7 (Float64)
relative for objectives.  The oracle runs one restart at a time (its BLAS calls are not safe to overlap in threads); where a
batch is too large for it, some restarts are checked against it and every restart against the scalar tiled pass
(engine = 4) or against the same restart solved alone."""
import math

import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu
SEED = 2015
EPS64 = float(np.finfo(np.float64).eps)
STOP = {"maxiter": 1, "tol": 2, "reattempts": 3}


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
    check (kl_tiled.cuh:959-1000 count them: sums + pass per half-update that runs, + the combine of a sliced one, + the
    image producer of the tc2 pass, + the impute kernel with NaN)."""
    def count(maxiter):
        b = ctx.batch(k, R)
        b.init_random(SEED)
        l0 = ctx.launches
        ctx.solve([b], nb.default_params(maxiter=maxiter, **params))
        b.close()
        return ctx.launches - l0
    return count(2) - count(1)


def residual_sums(X, W, H, w=1.0):
    """(sum of ((X - W H) w)^2, sum of (X - W H)^2) in Float64 over the entries of X that are not NaN, X's zeros counted as 0."""
    E = np.asarray(X, dtype=np.float64) - np.asarray(W, dtype=np.float64) @ np.asarray(H, dtype=np.float64)
    Ew = E * o._julia_weight(w if np.isscalar(w) else np.asarray(w, dtype=np.float64), *E.shape)
    keep = ~np.isnan(E)
    return float(np.sum(Ew[keep] ** 2)), float(np.sum(E[keep] ** 2))


def philox_factor(seed, shape):
    """The first numbers of Philox(key=seed) as a column-major matrix: a factor drawn alone (NMFkMultiplicative.jl:37-55)."""
    return np.random.Generator(np.random.Philox(key=seed)).random(shape[0] * shape[1]).reshape(shape, order="F")


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


# ---- 1. fixed factors on the tensor-core passes ---------------------------------------------------------------------------------
# id: n, m, k, R, dtype, fixed factor, launches an iteration, restarts checked against the oracle
FIXED = {
    "tc2_k16_Hfixed": (12000, 1000, 16, 16, np.float32, "H", 3, (0, 1, 15)),
    "gen1_k24_Wfixed": (20000, 512, 24, 8, np.float32, "W", 2 + 1, (0, 7)),
    "gen1_k24_Hfixed": (20000, 512, 24, 8, np.float32, "H", 2, (0, 7)),
    "dmma_k8_Wfixed": (40000, 600, 8, 8, np.float64, "W", 2 + 1, (0, 7)),
    "dmma_k8_Hfixed": (40000, 600, 8, 8, np.float64, "H", 2, (0, 7)),
}


def _plant_sub_eps(F, R, axis):
    """Fixed-factor entries of 0 and 1e-300 (below eps): one per 97 rows of W (columns of H), a different column (row) per
    restart, never a whole row (column), so W H stays positive."""
    for r in range(R):
        idx = np.arange(5, F.shape[1 + axis], 97)
        c0, c1 = r % F.shape[2 - axis], (r + 1) % F.shape[2 - axis]
        if axis == 0:
            F[r, idx, c0] = 0
            F[r, idx + 1, c1] = 1e-300
        else:
            F[r, c0, idx] = 0
            F[r, c1, idx + 1] = 1e-300


@pytest.mark.parametrize("case", list(FIXED))
def test_fixed_factor_on_tensor_passes(ctx, case):
    """R >= 8 restarts with one factor fixed, 10 iterations on the tensor-core pass the engine picks for the shape: the free
    factor and obj_ssq of the listed restarts match the oracle; every restart matches the scalar tiled pass (engine=4); the
    fixed factor comes back as max(F, eps) exactly (the check at iteration 10 clamps it, NMFkMultiplicative.jl:99-100)."""
    n, m, k, R, dt, fixed, per_it, probe = FIXED[case]
    X = synth.mixture(n, m, 8, seed=SEED, dtype=dt)
    W0, H0 = synth.philox_inits(SEED, R, n, k, m, dtype=dt)
    _plant_sub_eps(W0 if fixed == "W" else H0, R, 0 if fixed == "W" else 1)
    if fixed == "W":
        assert n * k >= 1 << 18  # wide_clamp off only because W is fixed (kl_tiled.cuh:1021)
    kw = dict(Wfixed=int(fixed == "W"), Hfixed=int(fixed == "H"), maxiter=10, normalize=0)
    ctx.set_X(X)
    out = solve(ctx, k, W0, H0, engine=2, **kw)
    ref4 = solve(ctx, k, W0, H0, engine=4, **kw)
    assert np.all(out["iters"] == 10) and np.all(out["stop_reason"] == 1), (out["iters"], out["stop_reason"])
    free, fix = ("H", "W") if fixed == "W" else ("W", "H")
    F0 = W0 if fixed == "W" else H0
    clamped = np.maximum(F0, dt(EPS64))
    assert np.array_equal(out[fix], clamped) and np.array_equal(ref4[fix], clamped)
    assert np.any(F0 < dt(EPS64)) and not np.array_equal(F0, clamped)
    e4 = max(relerr(out[free][r], ref4[free][r]) for r in range(R))
    assert e4 < ftol(dt), e4
    X64 = np.asfortranarray(X.astype(np.float64))
    err = []
    for r in probe:
        W, H, obj = o.nmf_multiplicative(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=10,
                                         Wfixed=fixed == "W", Hfixed=fixed == "H")
        ref = dict(W=W, H=H)
        assert np.array_equal(ref[fix], np.maximum(F0[r].astype(np.float64), EPS64))
        err.append((relerr(out[free][r], ref[free]), abs(out["obj_ssq"][r] - obj) / obj))
        assert err[-1][0] < ftol(dt) and err[-1][1] < otol(dt), (r, err[-1])
    print("%s: largest relative differences %s %.2e, obj_ssq %.2e; against engine=4 %.2e"
          % (case, free, max(e[0] for e in err), max(e[1] for e in err), e4))
    assert launches_per_iteration(ctx, k, R, engine=2, **{key: kw[key] for key in ("Wfixed", "Hfixed")}) == per_it


def test_caller_patterns_draw_the_free_factor(ctx):
    """NMFkProgressive's execute(X, nk, nNMF; seed, Hinit, Hfixed=true) and NMFkMapping's execute_run(...; seed, Winit,
    Wfixed=true) at scale (Float64, k = 16, DMMA pass): restart i's free factor is the first n k (k m) numbers of
    Philox(seed + i) for every restart, the fixed one is the caller's; the results equal the oracle's run of the same
    initialisations (10 iterations)."""
    n, m, k, R = 24000, 400, 16, 8
    X = synth.mixture(n, m, 8, seed=SEED)
    rng = np.random.Generator(np.random.Philox(key=SEED + 1000))
    Hfix = np.asfortranarray(rng.random((k, m)))
    Wfix = np.asfortranarray(rng.random((m, k)))  # for the transposed problem, m rows
    XT = np.asfortranarray(X.T)
    assert n * k * R > 4 * 148 * 16 * 256  # more numbers than one pass of the init grid draws
    # the draws themselves, before any iteration
    for Xc, Wi, Hi in ((X, None, np.broadcast_to(Hfix, (R, k, m))), (XT, np.broadcast_to(Wfix, (R, m, k)), None)):
        ctx.set_X(Xc)
        b = ctx.batch(k, R)
        b.set_init(Wi, Hi, SEED)
        g = b.get()
        b.close()
        for r in range(R):
            if Wi is None:
                assert np.array_equal(g["W"][r], philox_factor(SEED + r + 1, (n, k))) and np.array_equal(g["H"][r], Hfix), r
            else:
                assert np.array_equal(g["H"][r], philox_factor(SEED + r + 1, (k, n))) and np.array_equal(g["W"][r], Wfix), r
    # Hinit + Hfixed through execute_k (no signal reordering)
    Wg, Hg, fg, rg, ag = nb.execute_k(X, k, R, seed=SEED, Hinit=Hfix, Hfixed=True, maxiter=10, ctx=ctx)
    inits = [(philox_factor(SEED + i, (n, k)), Hfix.copy()) for i in range(1, R + 1)]
    Wo, Ho, fo, ro, ao = o.execute_k(X.copy(), k, R, inits=inits, Hfixed=True, maxiter=10)
    assert np.array_equal(Hg, np.maximum(Hfix, EPS64)) and np.array_equal(Ho, Hg)
    e1 = (relerr(Wg, Wo), abs(fg - fo) / fo)
    assert e1[0] < 1e-9 and e1[1] < 1e-7 and abs(rg - ro) < 1e-8 and abs(ag - ao) <= X.size * 1e-9, (e1, rg, ro, ag, ao)
    assert launches_per_iteration(ctx, k, R, Hfixed=1) == 2
    # Winit + Wfixed through execute_run on the transposed matrix (H drawn: k x 24000 per restart)
    Wg, Hg, fg, rg, ag = nb.execute_run(XT, k, R, seed=SEED, Winit=Wfix, Wfixed=True, maxiter=10, ctx=ctx)
    inits = [(Wfix.copy(), philox_factor(SEED + i, (k, n))) for i in range(1, R + 1)]
    Wo, Ho, fo, ro, ao = o.execute_run(XT.copy(), k, R, inits=inits, Wfixed=True, maxiter=10)
    assert np.array_equal(Wg, np.maximum(Wfix, EPS64)) and np.array_equal(Wo, Wg)
    e2 = (relerr(Hg, Ho), abs(fg - fo) / fo)
    assert e2[0] < 1e-9 and e2[1] < 1e-7 and abs(rg - ro) < 1e-8 and abs(ag - ao) <= X.size * 1e-9, (e2, rg, ro, ag, ao)
    assert launches_per_iteration(ctx, k, R, Wfixed=1) == 2
    print("caller patterns: Hfixed W %.2e fit %.2e; Wfixed H %.2e fit %.2e" % (e1 + e2))


# ---- 2. weights with the full stop rule -------------------------------------------------------------------------------------------
WN, WM, WR, WPROBE = 3000, 1000, 16, (0, 15)
WCASES = {"f32_k8_tc2": (np.float32, 8, 4 + 3), "f32_k20_gen1": (np.float32, 20, 3 + 2), "f64_k8_dmma": (np.float64, 8, 3 + 2)}
WRULE = dict(maxiter=40, maxbaditers=2, maxreattempts=1)


def replay_stop(objs, tol, tolOF, maxiter=40, maxbad=2, maxre=1):
    """The stop machine of nmf_multiplicative (oracle :174-224, checks every 10 iterations) replayed on a sequence of check
    objectives -> (iterations, reason, relative distances of every decision from its threshold)."""
    best, bad, re, margin = math.inf, 0, 0, []
    for it in range(10, maxiter + 1, 10):
        obj = objs[it]
        margin.append(abs(obj / tol - 1))
        if obj < tol:
            return it, "tol", margin
        if obj < best:
            if best < math.inf:
                margin.append(abs((best - obj) / tolOF - 1))
            bad = bad + 1 if best - obj < tolOF else 0
            best = obj
        else:
            bad += 1
        if bad >= maxbad:
            re, bad = re + 1, 0
        if re >= maxre and it < maxiter:
            return it, "reattempts", margin
    return maxiter, "maxiter", margin


@pytest.fixture(scope="module")
def wdata():
    """X (Float32 values, 1 % zeros), the inits, the weights (Float32 values in [1, 2)) and, per k, the oracle's trajectory of the
    probed restarts: W, H after the checks at 10, 20, 30, 40 (the weight only enters the objective, so one trajectory serves
    every weight; a run stops at one of these checks)."""
    X = synth.mixture(WN, WM, 8, seed=SEED, dtype=np.float32)
    rng = np.random.Generator(np.random.Philox(key=SEED + 2))
    X[rng.random((WN, WM)) < 0.01] = 0
    X64 = np.asfortranarray(X.astype(np.float64))
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    weights = {"scalar": 2.0, "rows": f32(1 + rng.random(WN)), "cols": f32(1 + rng.random((1, WM))), "matrix": f32(1 + rng.random((WN, WM)))}
    traj = {}

    def trajectory(k):
        if k not in traj:
            W0, H0 = synth.philox_inits(SEED, WR, WN, k, WM, dtype=np.float32)
            traj[k] = dict(W0=W0, H0=H0, at={})
            for r in WPROBE:
                at = {}

                def tr(it, W, H, obj):
                    if it % 10 == 0:
                        at[it] = (W.copy(), H.copy())
                o.nmf_multiplicative(X64, k, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=40, trace=tr)
                traj[k]["at"][r] = at
        return traj[k]
    Xl = np.where(X64 == 0, 1e-32, X64)  # the matrix the checks see (:74): zeros substituted
    return dict(X=X, X64=X64, Xl=Xl, weights=weights, trajectory=trajectory)


def _choose_tol(objw, obj1):
    """tol and tolOF (candidates between neighbouring objectives / improvements of the probed restarts) such that every stop
    decision of the weighted and of the unweighted replay is at least 5 % from its threshold and the weight changes the stop
    of at least one probed restart; among those, one where the weighted run stops before maxiter, on tolOF if possible."""
    vals = sorted(v for objs in list(objw.values()) + list(obj1.values()) for v in objs.values())
    tols = [math.sqrt(a * b) for a, b in zip(vals, vals[1:]) if b > a * 1.11]
    imp = sorted(abs(objs[it - 10] - objs[it]) for objs in list(objw.values()) + list(obj1.values()) for it in (20, 30, 40))
    tofs = [math.sqrt(a * b) for a, b in zip(imp, imp[1:]) if b > a * 1.11] + [1e-3]
    best, score = None, -1
    for tolOF in tofs:
        for tol in tols:
            rw = {r: replay_stop(objw[r], tol, tolOF) for r in objw}
            r1 = {r: replay_stop(obj1[r], tol, tolOF) for r in obj1}
            if min(min(x[2]) for x in list(rw.values()) + list(r1.values())) < 0.05:
                continue
            if all(rw[r][:2] == r1[r][:2] for r in rw):
                continue
            s = 2 * any(x[1] == "reattempts" for x in rw.values()) + any(x[1] != "maxiter" for x in rw.values())
            if s > score:
                best, score = (tol, tolOF, rw, r1), s
    assert best is not None
    return best


@pytest.mark.parametrize("kind", ["scalar", "rows", "cols", "matrix"])
@pytest.mark.parametrize("case", list(WCASES))
def test_weights_with_the_stop_rule(ctx, wdata, case, kind):
    """A weight (scalar 2, or Float32 values in [1, 2) per row, column or entry) with the stop rule in full: iteration counts
    and stop reasons of the probed restarts equal the oracle's (its stop machine on its own trajectory, with tol and tolOF
    chosen at least 5 % from every decision, and such that the weight moves a stop); their factors match the oracle's at that
    stop.  Every restart stops like the scalar tiled pass and matches its factors.  obj_ssq is the weighted sum
    recomputed in Float64 from the returned factors (zeros of X count as 0), obj_norm the unweighted norm."""
    dt, k, per_it = WCASES[case]
    w = wdata["weights"][kind]
    tj = wdata["trajectory"](k)
    Xl = wdata["Xl"]
    objw, obj1 = {}, {}
    for r in WPROBE:
        objw[r], obj1[r] = {}, {}
        for it, (W, H) in tj["at"][r].items():
            objw[r][it], obj1[r][it] = residual_sums(Xl, W, H, w)
    tol, tolOF, rw, r1 = _choose_tol(objw, obj1)
    X, W0, H0 = wdata["X"].astype(dt), tj["W0"].astype(dt), tj["H0"].astype(dt)
    ctx.set_X(X)
    scalar = np.isscalar(w)
    try:
        ctx.set_weight(None if scalar else w)
        p = dict(WRULE, tol=tol, tolOF=tolOF, weight=w if scalar else 1.0, normalize=0)
        out = solve(ctx, k, W0, H0, engine=2, **p)
        ref4 = solve(ctx, k, W0, H0, engine=4, **p)
        per = launches_per_iteration(ctx, k, WR, engine=2, normalize=0)
    finally:
        ctx.set_weight(None)
    assert np.array_equal(out["iters"], ref4["iters"]) and np.array_equal(out["stop_reason"], ref4["stop_reason"]), (out, ref4)
    e4 = max(max(relerr(out["W"][r], ref4["W"][r]), relerr(out["H"][r], ref4["H"][r])) for r in range(WR))
    assert e4 < ftol(dt), e4
    err = []
    for r in WPROBE:
        it, why, _ = rw[r]
        assert (out["iters"][r], out["stop_reason"][r]) == (it, STOP[why]), (r, out["iters"][r], out["stop_reason"][r], rw[r], r1[r])
        W, H = tj["at"][r][it]
        ow = residual_sums(wdata["X64"], W, H, w)[0]  # the oracle's :125
        err.append((relerr(out["W"][r], W), relerr(out["H"][r], H), abs(out["obj_ssq"][r] - ow) / ow))
        assert err[-1][0] < ftol(dt) and err[-1][1] < ftol(dt) and err[-1][2] < otol(dt), (r, err[-1])
    dobj = 0.0
    for r in range(WR):
        sw, s1 = residual_sums(wdata["X64"], out["W"][r], out["H"][r], w)
        dobj = max(dobj, abs(out["obj_ssq"][r] - sw) / sw, abs(out["obj_norm"][r] - math.sqrt(s1)) / math.sqrt(s1))
    assert dobj < otol(dt), dobj
    print("weights %s %s: stops %s (weight 1: %s); largest relative differences W %.2e, H %.2e, obj_ssq %.2e; recomputed "
          "objectives %.2e; engine=4 %.2e" % (case, kind, [rw[r][:2] for r in WPROBE], [r1[r][:2] for r in WPROBE],
                                              max(e[0] for e in err), max(e[1] for e in err), max(e[2] for e in err), dobj, e4))
    assert per == per_it, per


# ---- 3. normalizevector -----------------------------------------------------------------------------------------------------------
NVN, NVM, NVR, NVPROBE = 2500, 1012, 8, (0, 7)  # multiples of 4, not of 32
NVBLEND = (2, 5)  # the resume test starts them from blends of the mixture's own factors: they stop on tol at 10
NVCASES = {"f32_k8_tc2": (np.float32, 8, 4 + 3, False), "f32_k20_gen1": (np.float32, 20, 3 + 2, False),
           "f64_k8_dmma": (np.float64, 8, 3 + 2, False), "f64_k8_dmma_rowweight": (np.float64, 8, 3 + 2, True)}


@pytest.fixture(scope="module")
def nvdata():
    X = synth.mixture(NVN, NVM, 8, seed=SEED, dtype=np.float32)
    rng = np.random.Generator(np.random.Philox(key=SEED + 3))
    nv = (0.25 + rng.random(NVN)).astype(np.float32)
    wrow = (1 + rng.random(NVN)).astype(np.float32)
    X64 = np.asfortranarray(X.astype(np.float64))
    assert np.min(X64) > 0
    cache = {}

    def oracle(k, r, W0, H0, weight=1, **kw):
        key = (k, r, np.isscalar(weight), tuple(sorted(kw.items())))
        if key not in cache:
            objs = {}

            def tr(it, W, H, obj):
                if obj is not None:
                    objs[it] = obj
            inf = {}
            W, H, phi = o.execute_singlerun_compute(X64.copy(order="F"), k, Winit=W0.astype(np.float64), Hinit=H0.astype(np.float64),
                                                    normalizevector=nv.astype(np.float64), weight=weight, trace=tr, info=inf, **kw)
            cache[key] = dict(W=W, H=H, phi=phi, objs=objs, info=inf)
        return cache[key]
    return dict(X=X, X64=X64, nv=nv, wrow=wrow.astype(np.float64), oracle=oracle)


@pytest.mark.parametrize("case", list(NVCASES))
def test_normalizevector_batch(ctx, nvdata, case):
    """A batch of 8 restarts on X ./ nv, 20 iterations, normalize=1: restarts 0 and 7 match
    execute_singlerun_compute(...; normalizevector=nv) (W scaled back, rows of H summing to one, the norm against the caller's
    X); every restart's obj_ssq is the (weighted) sum against X recomputed from its returned factors."""
    dt, k, per_it, weighted = NVCASES[case]
    X, nv = nvdata["X"].astype(dt), nvdata["nv"].astype(dt)
    W0, H0 = synth.philox_inits(SEED, NVR, NVN, k, NVM, dtype=np.float32)
    w = nvdata["wrow"] if weighted else 1.0
    ctx.set_X(X, normalizevector=nv)
    try:
        ctx.set_weight(w if weighted else None)
        out = solve(ctx, k, W0.astype(dt), H0.astype(dt), maxiter=20, engine=2, normalize=1)
        per = launches_per_iteration(ctx, k, NVR, engine=2, normalize=1)
    finally:
        ctx.set_weight(None)
    assert np.all(out["iters"] == 20) and np.all(out["stop_reason"] == 1)
    err = []
    for r in NVPROBE:
        ref = nvdata["oracle"](k, r, W0[r], H0[r], weight=w, maxiter=20)
        err.append((relerr(out["W"][r], ref["W"]), relerr(out["H"][r], ref["H"]), abs(out["obj_norm"][r] - ref["phi"]) / ref["phi"]))
        assert err[-1][0] < ftol(dt) and err[-1][1] < ftol(dt) and err[-1][2] < otol(dt), (r, err[-1])
    dobj = 0.0
    for r in range(NVR):
        assert np.allclose(out["H"][r].astype(np.float64).sum(axis=1), 1.0, rtol=0, atol=1e-5 if dt == np.float32 else 1e-12), r
        sw, s1 = residual_sums(nvdata["X64"], out["W"][r], out["H"][r], w)
        dobj = max(dobj, abs(out["obj_ssq"][r] - sw) / sw, abs(out["obj_norm"][r] - math.sqrt(s1)) / math.sqrt(s1))
    assert dobj < otol(dt), dobj
    print("normalizevector %s: largest relative differences W %.2e, H %.2e, obj_norm %.2e; recomputed objectives %.2e"
          % ((case,) + tuple(max(e[i] for e in err) for i in range(3)) + (dobj,)))
    assert per == per_it, per


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_normalizevector_clusterW_tall(ctx, dt):
    """execute_singlerun(...; clusterWmatrix=true, normalizevector=nv) on a tall matrix (n k >= 2^18), 20 iterations: W, H and
    the norm match the oracle, the columns of W sum to one."""
    n, m, k = 36004, 124, 8
    X = synth.mixture(n, m, 8, seed=SEED, dtype=np.float32)
    nv = (0.25 + np.random.Generator(np.random.Philox(key=SEED + 4)).random(n)).astype(np.float32)
    W0, H0 = synth.philox_inits(SEED, 1, n, k, m, dtype=np.float32)
    W, H, phi = nb.execute_singlerun(X.astype(dt), k, Winit=W0[0].astype(dt), Hinit=H0[0].astype(dt), clusterWmatrix=True,
                                     normalizevector=nv.astype(dt), maxiter=20, engine=2, ctx=ctx)
    Wo, Ho, phio = o.execute_singlerun_compute(np.asfortranarray(X.astype(np.float64)), k, Winit=W0[0].astype(np.float64),
                                               Hinit=H0[0].astype(np.float64), clusterWmatrix=True,
                                               normalizevector=nv.astype(np.float64), maxiter=20)
    e = (relerr(W, Wo), relerr(H, Ho), abs(float(phi) - phio) / phio)
    assert e[0] < ftol(dt) and e[1] < ftol(dt) and e[2] < otol(dt), e
    assert np.allclose(W.astype(np.float64).sum(axis=0), 1.0, rtol=0, atol=1e-4 if dt == np.float32 else 1e-12)
    print("normalizevector clusterWmatrix %s: relative differences W %.2e, H %.2e, objective %.2e" % ((np.dtype(dt).name,) + e))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_normalizevector_resume(ctx, nvdata, dt):
    """The batch of test_normalizevector_batch (k = 8) with restarts 2 and 5 started from blends of the mixture's factors and tol
    between their objective at 10 and that of the others: paused with iter_limit=10 (2 and 5 stop and are scaled back by nv in
    the first call) and resumed to maxiter=20, it equals the continuous run bit for bit; restart 2 matches the oracle."""
    k = 8
    X, nv = nvdata["X"], nvdata["nv"]
    W0, H0 = synth.philox_inits(SEED, NVR, NVN, k, NVM, dtype=np.float32)
    rng = np.random.Generator(np.random.Philox(key=SEED))  # the factors synth.mixture multiplied
    Wt, Ht = rng.random((NVN, 8)), rng.random((8, NVM))
    for r in NVBLEND:
        W0[r] = (0.5 * W0[r] + 0.5 * Wt / nv.astype(np.float64)[:, None]).astype(np.float32)
        H0[r] = (0.5 * H0[r] + 0.5 * Ht).astype(np.float32)
    orc = nvdata["oracle"]
    below = max(orc(k, r, W0[r], H0[r], maxiter=10)["objs"][10] for r in NVBLEND)
    above = min(orc(k, r, W0[r], H0[r], maxiter=20)["objs"][it] for r in NVPROBE for it in (10, 20))
    tol = math.sqrt(below * above)
    assert below < tol / 1.05 and above > tol * 1.05, (below, tol, above)
    ctx.set_X(X.astype(dt), normalizevector=nv.astype(dt))
    p = dict(maxiter=20, tol=tol, engine=2, normalize=1)
    cont = solve(ctx, k, W0.astype(dt), H0.astype(dt), **p)
    b = ctx.batch(k, NVR)
    b.set_init(W0.astype(dt), H0.astype(dt))
    ctx.solve([b], nb.default_params(iter_limit=10, **p))
    mid = b.get(factors=False)
    assert all(mid["stop_reason"][r] == 2 for r in NVBLEND) and all(mid["stop_reason"][r] == 0 for r in NVPROBE), mid["stop_reason"]
    ctx.solve([b], nb.default_params(**p))
    res = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    for key in ("iters", "stop_reason", "obj_ssq", "obj_norm", "W", "H"):
        assert np.array_equal(res[key], cont[key]), key
    ref = orc(k, 2, W0[2], H0[2], maxiter=20, tol=tol)
    assert ref["info"]["iters"] == 10 and ref["info"]["stop_reason"] == "tol" and res["iters"][2] == 10
    e = (relerr(res["W"][2], ref["W"]), relerr(res["H"][2], ref["H"]), abs(res["obj_norm"][2] - ref["phi"]) / ref["phi"])
    assert e[0] < ftol(dt) and e[1] < ftol(dt) and e[2] < otol(dt), e


# ---- 4. missing entries at scale --------------------------------------------------------------------------------------------------
NAN_N, NAN_M, NAN_K, NAN_R, NAN_PROBE, NAN_AT = 8192, 1024, 12, 8, (0, 7), (1, 10, 20)


@pytest.fixture(scope="module")
def nandata():
    """X with 5 % NaN and 1 % zeros (Float32 values, so one oracle run serves both types) and the oracle's W, H of restarts 0
    and 7 after iterations 1, 10 and 20, with its final objective (:125, NaN entries left out)."""
    X = synth.mixture(NAN_N, NAN_M, 8, seed=SEED, dtype=np.float32)
    rng = np.random.Generator(np.random.Philox(key=SEED + 5))
    u = rng.random((NAN_N, NAN_M))
    X[u < 0.05] = np.nan
    X[(u >= 0.05) & (u < 0.06)] = 0
    W0, H0 = synth.philox_inits(SEED, NAN_R, NAN_N, NAN_K, NAN_M, dtype=np.float32)
    X64 = np.asfortranarray(X.astype(np.float64))
    ref = {}
    for r in NAN_PROBE:
        at = {}

        def tr(it, W, H, obj):
            if it in NAN_AT:
                at[it] = (W.copy(), H.copy())
        _, _, obj = o.nmf_multiplicative(X64, NAN_K, Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), maxiter=20, trace=tr)
        ref[r] = dict(at=at, obj=obj)
    assert np.isnan(X64).any() and np.sum(X64 == 0) > 0  # X64 comes back restored
    return dict(X=X, X64=X64, W0=W0, H0=H0, ref=ref)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_missing_entries_at_scale(ctx, nandata, dt):
    """8 restarts on X with NaN and zeros (the scalar HASNAN pass with both half-updates sliced): restarts 0 and 7 match the
    oracle after 1, 10 and 20 iterations; every restart matches the same restart solved alone (R = 1: other slice counts, its
    own imputation store); obj_ssq leaves out the NaN entries; a run paused at 10 and resumed equals the continuous run bit
    for bit."""
    X, W0, H0 = nandata["X"].astype(dt), nandata["W0"].astype(dt), nandata["H0"].astype(dt)
    ctx.set_X(X)
    assert ctx.xinfo().nnan > 0
    p = dict(engine=2, normalize=0)
    err = []
    for it in NAN_AT:
        out = solve(ctx, NAN_K, W0, H0, maxiter=it, **p)
        assert np.all(out["iters"] == it) and np.all(out["stop_reason"] == 1)
        for r in NAN_PROBE:
            W, H = nandata["ref"][r]["at"][it]
            err.append((relerr(out["W"][r], W), relerr(out["H"][r], H)))
            assert err[-1][0] < ftol(dt) and err[-1][1] < ftol(dt), (it, r, err[-1])
    cont = out  # 20 iterations
    dobj = 0.0
    for r in NAN_PROBE:
        ref = nandata["ref"][r]["obj"]
        dobj = max(dobj, abs(cont["obj_ssq"][r] - ref) / ref)
    for r in range(NAN_R):
        sw, s1 = residual_sums(nandata["X64"], cont["W"][r], cont["H"][r])
        dobj = max(dobj, abs(cont["obj_ssq"][r] - sw) / sw, abs(cont["obj_norm"][r] - math.sqrt(s1)) / math.sqrt(s1))
    assert dobj < otol(dt), dobj
    e1 = 0.0
    for r in range(NAN_R):
        one = solve(ctx, NAN_K, W0[r:r + 1], H0[r:r + 1], maxiter=20, **p)
        e1 = max(e1, relerr(cont["W"][r], one["W"][0]), relerr(cont["H"][r], one["H"][0]))
    assert e1 < ftol(dt), e1
    b = ctx.batch(NAN_K, NAN_R)
    b.set_init(W0, H0)
    ctx.solve([b], nb.default_params(maxiter=20, iter_limit=10, **p))
    assert np.all(b.get(factors=False)["stop_reason"] == 0)
    ctx.solve([b], nb.default_params(maxiter=20, **p))
    res = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    for key in ("iters", "stop_reason", "obj_ssq", "obj_norm", "W", "H"):
        assert np.array_equal(res[key], cont[key]), key
    print("missing entries %s: largest relative differences W %.2e, H %.2e, objectives %.2e; R = 8 against R = 1 %.2e"
          % (np.dtype(dt).name, max(e[0] for e in err), max(e[1] for e in err), dobj, e1))
    assert launches_per_iteration(ctx, NAN_K, NAN_R, **p) == 3 + 3 + 1
    assert launches_per_iteration(ctx, NAN_K, 1, **p) == 3 + 3 + 1
