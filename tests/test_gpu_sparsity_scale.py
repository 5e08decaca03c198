"""NMFsparsity (method=:sparsity, nmfk.jl_b200/csrc/sparsity.cu) against the Float64 oracle (oracle.nmf_sparsity) at the sizes users
run: restart batches, every beta mode in both precisions, k up to 32, exact zeros in X, paused and resumed runs, several batches
in one solve, and the execute / execute_run decisions.  Data and initial factors are drawn in Float32, so one oracle run serves
both precisions (except at the C4 shape, which is Float64).

  test                                    shape, batch                      branches reached (sparsity.cu)
  test_beta_modes_ragged                  2053 x 1031, R=16, 25 it.,        sp_pass_kernel / sp_objective_kernel with a partial
                                          tol=0; ed k=8, kl k=9, is k=16,   last CTA (2053 = 16 x 128 + 5 rows, 1031 = 8 x 128 + 7
                                          beta=1.5 k=17, beta=0.5 k=32;     columns) and SP_TT tails (1031 = 32 x 32 + 7, 2053 =
                                          f32 and f64                       64 x 32 + 5); every bmode of sp_terms and of the
                                                                            objective; KMAX = 8, 16 (k = 9, 16) and 32 (k = 17, 32)
                                                                            in both types; blockIdx.y up to 15; restarts 0, 7, 15
  test_c3_shape_ed                        10000^2 f32 k=16 R=64 ed, 3 it.   79 CTAs along each side with a 16-row tail, 64 restarts
                                                                            in the grid's y; restarts 0, 33, 63
  test_c4_shape_kl                        100000 x 2000 f64 k=32 R=64 kl,   the H half reduces over 100 000 rows in the KMAX = 32
                                          3 it.                             Float64 kernel; restarts 0, 63
  test_stop_rule_in_batch                 300 x 120, k=5, R=32, maxiter=37  sp_state_kernel stops restarts at iterations that are
                                                                            not multiples of check_every while tiled_guard_kernel
                                                                            only runs every 10; stopped restarts sit frozen
  test_exact_zeros                        200 x 80 with 10 % zeros (one     zeros of X substituted by nmfk_set_X count as 0 in
                                          whole row and column), k=4        sp_pass_kernel and sp_objective_kernel: kl and is
                                                                            objectives are NaN / Inf and run to maxiter
  test_resume_equals_continuous           the stop-rule batch, paused at    solve_sparsity_t skips the initial column normalisation
                                          every iteration                   on a resume and carries last_of in UnitState::best
  test_batch_composition                  the stop-rule batch; k = 5, 12,   per-restart kernels (nothing depends on R); three
                                          24 in one solve                   batches of different KMAX one after the other, each with
                                                                            its own scratch
  test_execute_run_sparsity               600 x 200 f64, k=4, R=32          nmfk_execute_run and the composed path with variant 2
  test_execute_sparsity_decisions         600 x 200 f64, ks=2:6, R=16       nmfk_execute: five batches in one nmfk_solve
  test_refusals                           small                             solve_sparsity_batches (capi.cu) and
                                                                            nmfk_set_sparsity_options refusals

Tolerances are the scale files' defaults: 1e-9 (Float64) and 1e-4 (Float32) relative on factors, 1e-7 and 2e-3 relative on
objectives.  The oracle runs one restart at a time (concurrent oracle runs in threads of one process gave wrong factors: its
BLAS calls are not safe to overlap)."""
import math

import numpy as np
import pytest

import nmfk_b200 as nb
from nmfk_b200 import synth
from nmfk_b200._lib import NMFkError
from nmfk_b200.api import _params_from_kw
from oracle import nmfk_oracle as o

pytestmark = pytest.mark.gpu
SEED = 2015
CHECK_EVERY = 10  # nmfk_params.check_every: tiled_guard_kernel runs after every 10th iteration
E_INVALID, E_UNSUPPORTED = -1, -6


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def ftol(dt):
    return 1e-9 if dt == np.float64 else 1e-4


def otol(dt):
    return 1e-7 if dt == np.float64 else 2e-3


def sp_params(ctx, cost_function="ed", beta_divergence=-1, sparsity=1.0, **p):
    """nmfk_params of method=:sparsity; the NMFsparsity options go to the context (nmfk_set_sparsity_options)."""
    p.setdefault("normalize", 0)
    return _params_from_kw(dict(method="sparsity", cost_function=cost_function, beta_divergence=beta_divergence, sparsity=sparsity),
                           ctx, **p)


def solve(ctx, k, W0, H0, params):
    b = ctx.batch(k, W0.shape[0])
    b.set_init(W0, H0)
    ctx.solve([b], params)
    out = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    return out


def oracle(X64, W0, H0, r, **kw):
    inf = {}
    W, H, ssq = o.nmf_sparsity(X64, W0.shape[2], Winit=W0[r].astype(np.float64), Hinit=H0[r].astype(np.float64), info=inf, **kw)
    return dict(W=W, H=H, ssq=ssq, info=inf)


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


# ---- 1. every beta mode at ragged mid-size shapes ------------------------------------------------------------------------------
RAG_N, RAG_M, RAG_R, RAG_IT = 2053, 1031, 16, 25
RAG_PROBE = (0, 7, 15)
# (cost_function, beta_divergence, k, sparsity): bmode 2, 1, 0 and the general pow() branch twice; KMAX 8, 16, 16, 32, 32
RAG_CASES = {"ed": ("ed", -1, 8, 0.5), "kl": ("kl", -1, 9, 0.0), "is": ("is", -1, 16, 0.1), "beta1.5": ("ed", 1.5, 17, 0.0),
             "beta0.5": ("ed", 0.5, 32, 0.3)}
_rag_cache = {}


def _ragged(case):
    if case not in _rag_cache:
        cf, beta, k, sp = RAG_CASES[case]
        X = synth.mixture(RAG_N, RAG_M, 6, seed=SEED, dtype=np.float32)
        W0, H0 = synth.philox_inits(SEED, RAG_R, RAG_N, k, RAG_M, dtype=np.float32)
        X64 = np.asfortranarray(X.astype(np.float64))
        ref = {r: oracle(X64, W0, H0, r, cost_function=cf, beta_divergence=beta, sparsity=sp, maxiter=RAG_IT, tol=0.0) for r in RAG_PROBE}
        _rag_cache[case] = dict(X=X, W0=W0, H0=H0, ref=ref)
    return _rag_cache[case]


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("case", list(RAG_CASES))
def test_beta_modes_ragged(ctx, case, dt):
    """25 iterations of 16 restarts with tol = 0: every restart stops on maxiter; restarts 0, 7 and 15 match the oracle in W, H
    and obj_ssq (sum((X - W*H)^2) of :109-110), and W keeps unit-norm columns (:86)."""
    cf, beta, k, sp = RAG_CASES[case]
    d = _ragged(case)
    ctx.set_X(d["X"].astype(dt))
    out = solve(ctx, k, d["W0"].astype(dt), d["H0"].astype(dt), sp_params(ctx, cf, beta, sp, maxiter=RAG_IT, tol=0.0))
    assert np.all(out["iters"] == RAG_IT) and np.all(out["stop_reason"] == 1), (out["iters"], out["stop_reason"])
    err = []
    for r in RAG_PROBE:
        ref = d["ref"][r]
        err.append((relerr(out["W"][r], ref["W"]), relerr(out["H"][r], ref["H"]), abs(out["obj_ssq"][r] - ref["ssq"]) / ref["ssq"]))
        assert err[-1][0] < ftol(dt) and err[-1][1] < ftol(dt) and err[-1][2] < otol(dt), (r, err[-1])
    for r in range(RAG_R):
        assert np.allclose(np.linalg.norm(out["W"][r].astype(np.float64), axis=0), 1.0, rtol=0, atol=1e-5 if dt == np.float32 else 1e-12), r
    print("ragged %s %s k=%d: largest relative differences W %.2e, H %.2e, obj_ssq %.2e"
          % ((case, np.dtype(dt).name, k) + tuple(max(e[i] for e in err) for i in range(3))))


# ---- 2. the benchmark's matrices -----------------------------------------------------------------------------------------------
def test_c3_shape_ed(ctx):
    """C3's matrix (10000 x 10000 Float32) with C3's batch (k = 16, 64 restarts), cost_function = ed, 3 iterations: restarts 0, 33
    and 63 against the oracle."""
    n, k, R, niter = 10000, 16, 64, 3
    X = synth.mixture(n, n, 16, seed=SEED, dtype=np.float32)
    W0, H0 = synth.philox_inits(SEED, R, n, k, n, dtype=np.float32)
    ctx.set_X(X)
    out = solve(ctx, k, W0, H0, sp_params(ctx, "ed", sparsity=1.0, maxiter=niter))
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1)
    X64 = np.asfortranarray(X.astype(np.float64))
    del X
    err = []
    for r in (0, 33, 63):
        ref = oracle(X64, W0, H0, r, cost_function="ed", sparsity=1.0, maxiter=niter)
        err.append((relerr(out["W"][r], ref["W"]), relerr(out["H"][r], ref["H"]), abs(out["obj_ssq"][r] - ref["ssq"]) / ref["ssq"]))
        assert err[-1][0] < 1e-4 and err[-1][1] < 1e-4 and err[-1][2] < 2e-3, (r, err[-1])
    print("C3 sparsity ed: largest relative differences W %.2e, H %.2e, obj_ssq %.2e" % tuple(max(e[i] for e in err) for i in range(3)))


def test_c4_shape_kl(ctx):
    """C4's matrix (100000 x 2000 Float64), k = 32, 64 restarts, kl, 3 iterations: restarts 0 and 63 against the oracle."""
    n, m, k, R, niter = 100000, 2000, 32, 64, 3
    X = synth.mixture(n, m, 8, seed=SEED, dtype=np.float64)
    W0, H0 = synth.philox_inits(SEED, R, n, k, m)
    ctx.set_X(X)
    out = solve(ctx, k, W0, H0, sp_params(ctx, "kl", sparsity=0.1, maxiter=niter))
    assert np.all(out["iters"] == niter) and np.all(out["stop_reason"] == 1)
    err = []
    for r in (0, 63):
        ref = oracle(X, W0, H0, r, cost_function="kl", sparsity=0.1, maxiter=niter)
        err.append((relerr(out["W"][r], ref["W"]), relerr(out["H"][r], ref["H"]), abs(out["obj_ssq"][r] - ref["ssq"]) / ref["ssq"]))
        assert err[-1][0] < 1e-9 and err[-1][1] < 1e-9 and err[-1][2] < 1e-7, (r, err[-1])
    print("C4 sparsity kl k=32: largest relative differences W %.2e, H %.2e, obj_ssq %.2e" % tuple(max(e[i] for e in err) for i in range(3)))


# ---- 3. the stop rule inside one batch -----------------------------------------------------------------------------------------
STOP_N, STOP_M, STOP_K, STOP_R, STOP_MAXITER, STOP_SP = 300, 120, 5, 32, 37, 0.1
STOP_EPS = 0.05  # Float32: the oracle's relative change at the deciding iterations is within 5 % of the device's
_stop_cache = {}


def _relchange(objs):
    """c[t] = |of(t) - of(t-1)| / of(t-1) for t = 2, ... (the test of :101-106); c[0] = c[1] = Inf."""
    c = np.full(len(objs) + 1, np.inf)
    for t in range(2, len(objs) + 1):
        c[t] = abs(objs[t - 1] - objs[t - 2]) / objs[t - 2]
    return c


def _stop_iter(c, tol, maxiter):
    hit = np.flatnonzero(c[2:maxiter + 1] < tol)
    return (int(hit[0]) + 2, "tol") if hit.size else (maxiter, "maxiter")


def _stop_case():
    """Float32 data, 32 restarts and the oracle's whole 37-iteration trace of each.  tol is the geometric mean of two adjacent
    relative changes of the trace, chosen so that the restarts stop on it at three or more different iterations, none a multiple
    of check_every, and as far as possible from every relative change that decides a stop."""
    if not _stop_cache:
        X = synth.mixture(STOP_N, STOP_M, 4, seed=SEED, dtype=np.float32)
        W0, H0 = synth.philox_inits(SEED, STOP_R, STOP_N, STOP_K, STOP_M, dtype=np.float32)
        X64 = np.asfortranarray(X.astype(np.float64))
        trace = []
        for r in range(STOP_R):
            tr = []
            oracle(X64, W0, H0, r, sparsity=STOP_SP, maxiter=STOP_MAXITER, tol=0.0,
                   trace=lambda it, W, H, of: tr.append((W.copy(), H.copy(), of)))
            trace.append(tr)
        crit = [_relchange([s[2] for s in tr]) for tr in trace]
        vals = np.unique(np.concatenate([c[2:] for c in crit]))
        best = None
        for lo, hi in zip(vals[:-1], vals[1:]):
            tol = math.sqrt(lo * hi)
            stops = [_stop_iter(c, tol, STOP_MAXITER) for c in crit]
            at = {t for t, why in stops if why == "tol"}
            if len(at) < 3 or any(t % CHECK_EVERY == 0 for t in at) or all(why == "tol" for _, why in stops):
                continue
            if best is None or hi / lo > best[0]:
                best = (hi / lo, tol, stops)
        assert best is not None
        _stop_cache.update(X=X, W0=W0, H0=H0, X64=X64, trace=trace, crit=crit, tol=best[1], margin=best[0], stops=best[2])
    return _stop_cache


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_stop_rule_in_batch(ctx, dt):
    """32 restarts with the relative-change stop rule (:101-106) and maxiter = 37: restarts stop on the tolerance at three or more
    different iterations between the guard's checks and the rest run to maxiter.  Float64: iteration counts and stop reasons
    equal the oracle's and W, H match its trace at the stop iteration.  Float32: the stop iteration t brackets the oracle's
    criterion, c(t) < tol (1 + eps) and c(t - 1) >= tol (1 - eps) with eps = STOP_EPS (no earlier t' has c(t') < tol (1 - eps)),
    and the factors match the oracle at t."""
    d = _stop_case()
    tol = d["tol"]
    ctx.set_X(d["X"].astype(dt))
    out = solve(ctx, STOP_K, d["W0"].astype(dt), d["H0"].astype(dt), sp_params(ctx, sparsity=STOP_SP, maxiter=STOP_MAXITER, tol=tol))
    reason = {"tol": 2, "maxiter": 1}
    err = []
    for r in range(STOP_R):
        t, why = int(out["iters"][r]), int(out["stop_reason"][r])
        c = d["crit"][r]
        if dt == np.float64:
            assert (t, why) == (d["stops"][r][0], reason[d["stops"][r][1]]), (r, t, why, d["stops"][r])
        elif why == 2:
            assert c[t] < tol * (1 + STOP_EPS) and c[t - 1] >= tol * (1 - STOP_EPS), (r, t, c[t - 2:t + 1] / tol)
            assert np.all(c[2:t] >= tol * (1 - STOP_EPS)), (r, t)
        else:
            assert (t, why) == (STOP_MAXITER, 1) and np.all(c[2:] >= tol * (1 - STOP_EPS)), (r, t, why)
        W, H, _ = d["trace"][r][t - 1]
        err.append(max(relerr(out["W"][r], W), relerr(out["H"][r], H)))
        assert err[-1] < ftol(dt), (r, t, err[-1])
    at = {int(t) for t, s in zip(out["iters"], out["stop_reason"]) if s == 2}
    assert len(at) >= 3 and all(t % CHECK_EVERY for t in at), (out["iters"], out["stop_reason"])
    print("stop rule %s: tol %.4e (gap %.4f), stop iterations %s, largest relative difference %.2e"
          % (np.dtype(dt).name, tol, d["margin"], sorted(at), max(err)))


# ---- 4. exact zeros in X -------------------------------------------------------------------------------------------------------
ZERO_N, ZERO_M, ZERO_K, ZERO_SP, ZERO_MAXITER = 200, 80, 4, 0.1, 220
ZERO_TOL = {"kl": 1e-3, "is": 1e-4, "ed": 1e-3}
_zero_cache = {}


def _zeros_case(cf):
    """X with its lowest 10 % of entries, row 17 and column 5 set to 0.  The oracle on X itself, and on X with the zeros replaced
    by 1e-32 (what nmfk_set_X leaves in the device's image of X): there kl and is stop on the tolerance well before maxiter."""
    if "X" not in _zero_cache:
        X = synth.mixture(ZERO_N, ZERO_M, 3, seed=SEED, dtype=np.float32)
        X[X <= np.quantile(X, 0.1)] = 0
        X[17, :] = 0
        X[:, 5] = 0
        W0, H0 = synth.philox_inits(SEED, 2, ZERO_N, ZERO_K, ZERO_M, dtype=np.float32)
        _zero_cache.update(X=X, W0=W0, H0=H0)
    if cf not in _zero_cache:
        X64 = np.asfortranarray(_zero_cache["X"].astype(np.float64))
        W0, H0 = _zero_cache["W0"], _zero_cache["H0"]
        kw = dict(cost_function=cf, sparsity=ZERO_SP, maxiter=ZERO_MAXITER, tol=ZERO_TOL[cf])
        with np.errstate(divide="ignore", invalid="ignore"):
            ref = oracle(X64, W0, H0, 0, **kw)
            sub = oracle(np.where(X64 == 0, 1e-32, X64), W0, H0, 0, **kw)
            tr = []  # every iteration up to maxiter, for the Float32 bracketing
            oracle(X64, W0, H0, 0, trace=lambda it, W, H, of: tr.append((W.copy(), H.copy(), of)), **dict(kw, tol=0.0))
        _zero_cache[cf] = dict(ref=ref, trace=tr, sub=sub)
    return _zero_cache, _zero_cache[cf]


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("cf", ["kl", "is", "ed"])
def test_exact_zeros(ctx, cf, dt):
    """Zeros of X count as zeros in the in-loop passes and objective, as in the reference, whose preprocessing is commented out:
    with kl the objective is NaN (0 log 0) and with is Inf (-log 0), the relative-change test is never true and the run goes to
    maxiter (stop reason 1), where the substituted 1e-32 would stop it on the tolerance early.  ed stops on the tolerance either
    way.  Iteration count and stop reason equal the oracle's (Float32 with ed: the bracketing check of test_stop_rule_in_batch);
    W, H match the oracle at that iteration."""
    z, d = _zeros_case(cf)
    inf, sub = d["ref"]["info"], d["sub"]["info"]
    if cf == "ed":
        assert inf["stop_reason"] == "tol" and inf["iters"] == sub["iters"], (inf, sub)
    else:  # the test is sensitive: substituting the zeros would stop the run early
        assert (inf["iters"], inf["stop_reason"]) == (ZERO_MAXITER, "maxiter") and not np.isfinite(inf["objective"]), inf
        assert sub["stop_reason"] == "tol" and sub["iters"] < ZERO_MAXITER // 2, sub
    ctx.set_X(z["X"].astype(dt))
    out = solve(ctx, ZERO_K, z["W0"][:1].astype(dt), z["H0"][:1].astype(dt),
                sp_params(ctx, cf, sparsity=ZERO_SP, maxiter=ZERO_MAXITER, tol=ZERO_TOL[cf]))
    t, why = int(out["iters"][0]), int(out["stop_reason"][0])
    if dt == np.float32 and cf == "ed":
        c = _relchange([s[2] for s in d["trace"]])
        tol = ZERO_TOL[cf]
        assert why == 2 and c[t] < tol * (1 + STOP_EPS) and np.all(c[2:t] >= tol * (1 - STOP_EPS)), (t, why, inf["iters"])
    else:
        assert (t, why) == (inf["iters"], 2 if inf["stop_reason"] == "tol" else 1), (t, why, inf, sub)
    W, H, _ = d["trace"][t - 1]
    e = (relerr(out["W"][0], W), relerr(out["H"][0], H))
    assert e[0] < ftol(dt) and e[1] < ftol(dt), e
    X64 = z["X"].astype(np.float64)
    ssq = float(np.sum((X64 - W @ H) ** 2))  # obj_ssq against the caller's X, zeros restored
    assert abs(out["obj_ssq"][0] - ssq) / ssq < otol(dt), (out["obj_ssq"][0], ssq)
    print("zeros %s %s: %d iterations (reason %d; with 1e-32: %d), relative differences W %.2e, H %.2e"
          % (cf, np.dtype(dt).name, t, why, sub["iters"], e[0], e[1]))


# ---- 5. a run paused at every iteration equals the continuous run --------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_resume_equals_continuous(ctx, dt):
    """The stop-rule batch solved with iter_limit = 1, 2, ..., 37 in 37 calls equals one 37-iteration call bit for bit (W, H after
    the normalisation, obj_norm, iterations, stop reasons).  After each pause p the restarts that stop on the tolerance at
    t <= p (before or at the pause) report stop reason 2, the others 0 (they stop after it)."""
    d = _stop_case()
    ctx.set_X(d["X"].astype(dt))
    W0, H0 = d["W0"].astype(dt), d["H0"].astype(dt)
    kw = dict(sparsity=STOP_SP, maxiter=STOP_MAXITER, tol=d["tol"], normalize=1)
    cont = solve(ctx, STOP_K, W0, H0, sp_params(ctx, **kw))
    stop_at = np.where(cont["stop_reason"] == 2, cont["iters"], STOP_MAXITER + 1)
    assert len(set(stop_at[stop_at <= STOP_MAXITER].tolist())) >= 3, cont["iters"]
    b = ctx.batch(STOP_K, STOP_R)
    b.set_init(W0, H0)
    for p in range(1, STOP_MAXITER):
        ctx.solve([b], sp_params(ctx, iter_limit=p, **kw))
        mid = b.get(factors=False)
        assert np.array_equal(mid["stop_reason"], np.where(stop_at <= p, 2, 0)), (p, mid["stop_reason"])
        assert np.array_equal(mid["iters"], np.minimum(stop_at, p)), (p, mid["iters"])
    ctx.solve([b], sp_params(ctx, iter_limit=STOP_MAXITER, **kw))
    res = {key: np.array(v) for key, v in b.get().items()}
    b.close()
    for key in ("iters", "stop_reason", "obj_ssq", "obj_norm", "W", "H"):
        assert np.array_equal(res[key], cont[key]), key


# ---- 6. batch composition ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_batch_composition(ctx, dt):
    """A restart solved alone equals the same restart inside the 32-restart batch bit for bit (every kernel works per restart),
    and three batches with k = 24, 5, 12 (KMAX 32, 8, 16) solved by one nmfk_solve call equal three separate calls bit for bit."""
    d = _stop_case()
    ctx.set_X(d["X"].astype(dt))
    W0, H0 = d["W0"].astype(dt), d["H0"].astype(dt)
    p = sp_params(ctx, sparsity=STOP_SP, maxiter=STOP_MAXITER, tol=d["tol"], normalize=1)
    full = solve(ctx, STOP_K, W0, H0, p)
    for r in (0, 13, STOP_R - 1):
        one = solve(ctx, STOP_K, W0[r:r + 1], H0[r:r + 1], p)
        for key in ("iters", "stop_reason", "obj_ssq", "obj_norm", "W", "H"):
            assert np.array_equal(one[key][0], full[key][r]), (r, key)
    inits = {}
    for k, R in ((24, 3), (5, 7), (12, 4)):
        inits[k] = synth.philox_inits(SEED + k, R, STOP_N, k, STOP_M, dtype=dt)
    p = sp_params(ctx, "kl", sparsity=0.05, maxiter=30, normalize=1)
    sep = {k: solve(ctx, k, *inits[k], p) for k in inits}
    bs = {}
    for k, (Wi, Hi) in inits.items():
        bs[k] = ctx.batch(k, Wi.shape[0])
        bs[k].set_init(Wi, Hi)
    ctx.solve(list(bs.values()), p)
    for k, b in bs.items():
        got = b.get()
        b.close()
        for key in ("iters", "stop_reason", "obj_ssq", "obj_norm", "W", "H"):
            assert np.array_equal(got[key], sep[k][key]), (k, key)


# ---- 7. execute_run and execute with method="sparsity" -------------------------------------------------------------------------
EX_N, EX_M, EX_MAXITER = 600, 200, 300
EX_KW = dict(method="sparsity", cost_function="kl", sparsity=0.05, maxiter=EX_MAXITER)


@pytest.fixture(scope="module")
def ex_data():
    X = synth.mixture(EX_N, EX_M, 4, seed=SEED) + 0.01
    return np.asfortranarray(X)


def test_execute_run_sparsity(ctx, ex_data):
    """execute_run(X, 4, 32; method=:sparsity) against the oracle's execute_run: the sort order of the restarts, the labels of the
    clustering, robustness, phi, AIC and the best W and H, through the one-call form (nmfk_execute_run) and the composed one."""
    X, k, R = ex_data, 4, 32
    W0, H0 = synth.philox_inits(SEED, R, EX_N, k, EX_M)
    det = {}
    Wo, Ho, phio, robo, aico = o.execute_run(X.copy(), k, R, inits=list(zip(W0, H0)), details=det, **EX_KW)
    assert all(s == "maxiter" for s in det["stop_reasons"])
    Wg, Hg, phi, rob, aic = nb.execute_run(X, k, R, inits=(W0, H0), ctx=ctx, **EX_KW)
    dg = {}
    Wc, Hc, phic, robc, aicc = nb.execute_run(X, k, R, inits=(W0, H0), ctx=ctx, details=dg, **EX_KW)
    assert np.array_equal(dg["order"], det["idxsort"]) and np.array_equal(dg["labels"], det["labels"]), (dg["order"], det["idxsort"])
    assert relerr(dg["fit"], det["objvalue"]) < 1e-7 and np.all(dg["iters"] == EX_MAXITER)
    for W, H, ph, rb, ac in ((Wg, Hg, phi, rob, aic), (Wc, Hc, phic, robc, aicc)):
        assert relerr(W, Wo) < 1e-9 and relerr(H, Ho) < 1e-9, (relerr(W, Wo), relerr(H, Ho))
        assert abs(ph - phio) / phio < 1e-7 and abs(rb - robo) < 1e-9 and abs(ac - aico) <= 1e-7 * abs(aico), (ph, phio, rb, robo, ac, aico)
    print("execute_run sparsity: robustness %.4f, phi %.2e / %.2e, AIC %.6g / %.6g" % (robo, phi, phio, aic, aico))


def test_execute_sparsity_decisions(ctx, ex_data):
    """execute(X, 2:6, 16; method=:sparsity) against the oracle's execute: kopt, fitquality, robustness and AIC for every k."""
    X, R, ks = ex_data, 16, range(2, 7)
    inits = {k: synth.philox_inits(SEED + k, R, EX_N, k, EX_M) for k in ks}
    _, _, fito, robo, aico, kopto = o.execute(X.copy(), ks, R, per_k_kw=lambda k: dict(inits=list(zip(*inits[k]))), **EX_KW)
    _, _, fit, rob, aic, kopt = nb.execute(X, ks, R, inits=inits, ctx=ctx, **EX_KW)
    assert kopt == kopto, (kopt, kopto, rob, robo)
    for k in ks:
        assert abs(fit[k - 1] - fito[k - 1]) / fito[k - 1] < 1e-7, (k, fit[k - 1], fito[k - 1])
        assert abs(rob[k - 1] - robo[k - 1]) < 1e-9, (k, rob[k - 1], robo[k - 1])
        assert abs(aic[k - 1] - aico[k - 1]) <= 1e-7 * abs(aico[k - 1]), (k, aic[k - 1], aico[k - 1])
    print("execute sparsity: kopt %s, robustness %s" % (kopt, np.round(robo[1:], 4)))


# ---- 8. refusals ---------------------------------------------------------------------------------------------------------------
def test_refusals(ctx):
    """NMFsparsity refuses X with NaN, k > 32, array weights and a normalizevector with NMFK_E_UNSUPPORTED and a message naming
    the reason; a non-positive lambda with NMFK_E_INVALID."""
    X = synth.mixture(64, 40, 3, seed=SEED) + 0.01

    def refused(status, words, k=4, **kw):
        with pytest.raises(NMFkError) as e:
            nb.NMFsparsity(Xs, k, ctx=ctx, maxiter=2, **kw)
        assert e.value.status == status and all(w in str(e.value) for w in words), str(e.value)

    Xs = X.copy()
    Xs[3, 7] = np.nan
    refused(E_UNSUPPORTED, ("NMFsparsity", "NaN"))
    Xs = X
    refused(E_UNSUPPORTED, ("NMFsparsity", "k > 32"), k=33)
    refused(E_INVALID, ("lambda must be positive",), lam=0.0)
    for kw in (dict(weight=np.linspace(0.5, 1.5, 64)), dict(normalizevector=np.linspace(1, 2, 64))):
        b = None
        with pytest.raises(NMFkError) as e:
            ctx.set_X(X, normalizevector=kw.get("normalizevector"))
            p = _params_from_kw(dict(method="sparsity", weight=kw.get("weight", 1)), ctx, maxiter=2)
            b = ctx.batch(3, 2)
            b.init_random(1)
            ctx.solve([b], p)
        if b is not None:
            b.close()
        assert e.value.status == E_UNSUPPORTED and "normalizevector and array weights" in str(e.value), str(e.value)
    ctx.set_weight(None)
    ctx.set_X(X)
    W, H, _ = nb.NMFsparsity(X, 32, ctx=ctx, maxiter=2)  # k = 32 is the largest accepted
    assert W.shape == (64, 32) and np.all(np.isfinite(H))
