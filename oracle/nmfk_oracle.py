"""CPU oracle: a NumPy restatement of the NMFk.jl factorization hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product: only
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` may import it, and there only as the checker or as the timed CPU
baseline.  The product path (``nmfk.jl_b200/``) never imports this module and fails loudly
when its CUDA library is missing.

PARITY PINNING STATUS ("parity unpinned" for per-iteration values):
  The reference is 100 % Julia and no Julia runtime exists in this image or on the GPU box,
  so the reference itself cannot be executed, and its own tests hold no numeric fixtures for
  this path (SURVEY.md §4).  What *is* pinned (tests/test_oracle_known_answers.py):
    * the recorded outputs of the reference on the blind-source-separation notebook
      (`notebooks/blind_source_separation/blind_source_separation.md:170-264`): X is printed
      there to 6 digits; the k=2 fit 13.93858 / silhouette 0.994 / AIC -46.21 and kopt = 3
      are reproduced by this oracle from its own random initialisations;
    * the feature-extraction notebook decision kopt = 4
      (`notebooks/feature_extraction/feature_extraction.md:208-292`);
    * the invariants asserted by `test/test_execute_smoke.jl:6-32`,
      `test/test_cluster_unit.jl:36-54`, `test/test_normalize.jl:44-55`,
      `test/test_helpers.jl:60-67`.
  Per-iteration W/H/fit values are NOT pinned by any reference artefact; they are defined by
  this restatement (Float64, NumPy/OpenBLAS summation order).

Every function cites the reference file:line it follows (paths relative to /root/reference).
Third-party semantics that are not vendored in the reference tree are restated from the
published packages and named where used:
  * Distances.jl (compat 0.8-0.11, Project.toml:63): ``cosine_dist``, ``pairwise(CosineDist())``
  * Clustering.jl (compat 0.14/0.15, Project.toml:55): ``silhouettes(assignments, dists)``
"""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import numpy as np

EPS64 = float(np.finfo(np.float64).eps)  # Julia `eps()` == eps(Float64), used for any T


# --------------------------------------------------------------------------------------
# Helpers: src/NMFkHelpers.jl
# --------------------------------------------------------------------------------------
def normnan(X: np.ndarray) -> float:
    """`normnan` src/NMFkHelpers.jl:226-228 : LinearAlgebra.norm(X[.!isnan.(X)])."""
    v = np.asarray(X)[~np.isnan(X)]
    r = np.sqrt(np.sum(v.astype(np.float64) ** 2))
    return float(np.float32(r)) if v.dtype == np.float32 else float(r)


def ssqrnan(X: np.ndarray) -> float:
    """`ssqrnan` src/NMFkHelpers.jl:222-224 : sum(X[.!isnan.(X)].^2)."""
    v = np.asarray(X)[~np.isnan(X)]
    return float(np.sum(v ** 2))


def zerostoepsilon(X: np.ndarray) -> np.ndarray:
    """`zerostoepsilon` src/NMFkHelpers.jl:529-543 : x < eps(T)^2 -> eps(T)^2 (copy)."""
    Xn = np.array(X, copy=True)
    e = np.finfo(Xn.dtype).eps ** 2
    Xn[Xn < e] = e
    return Xn


# --------------------------------------------------------------------------------------
# Solver: src/NMFkMultiplicative.jl
# --------------------------------------------------------------------------------------
class NegativeEntriesError(ValueError):
    """ErrorException("All matrix entries must be nonnegative!") NMFkMultiplicative.jl:4-7."""


def nmf_preprocessing(X: np.ndarray, lam: float = 1e-32):
    """`NMFpreprocessing!` src/NMFkMultiplicative.jl:3-22.  Mutates X, returns (inan, izero).

    `minimum(X)` propagates NaN in Julia (so does np.min), hence negative entries go
    undetected when X also holds NaNs - kept as is.
    """
    if X.size and np.min(X) < 0:
        raise NegativeEntriesError("All matrix entries must be nonnegative!")
    izero = X <= 0
    X[izero] = lam
    inan = np.isnan(X)
    X[inan] = lam
    return inan, izero


def _julia_weight(weight, n: int, m: int):
    """`(X - W*H) .* weight` under Julia's broadcasting: a Vector of length n is an n x 1 column (one weight per ROW),
    a 1 x m matrix weights the columns, an n x m matrix weights entries (the shapes execute_run asserts,
    src/NMFkExecute.jl:484).  NumPy would broadcast a 1-D array along the last axis, hence this helper."""
    if np.isscalar(weight):
        return weight
    w = np.asarray(weight)
    if w.ndim == 1:
        assert w.shape[0] == n, "length(weight) == size(X, 1)"
        return w.reshape(n, 1)
    assert w.shape in ((n, 1), (1, m), (n, m))
    return w


def _canon_partition(index: np.ndarray) -> np.ndarray:
    """Canonical form of the co-clustering matrix `cons` (NMFkMultiplicative.jl:105):
    cons[i,j] = (index[i]==index[j]) is determined by, for every column, the first column
    that shares its argmin."""
    first = {}
    out = np.empty(len(index), dtype=np.int64)
    for q, a in enumerate(index):
        out[q] = first.setdefault(int(a), q)
    return out


def nmf_multiplicative(
    X: np.ndarray,
    k: int,
    *,
    weight=1,
    tol: float = 1e-19,
    tolOF: float = 1e-3,
    lam: float = 1e-32,
    maxreattempts: int = 2,
    maxbaditers: int = 10,
    maxiter: int = 1000000,
    stopconv: int = 1000,
    Wfixed: bool = False,
    Hfixed: bool = False,
    Winit: Optional[np.ndarray] = None,
    Hinit: Optional[np.ndarray] = None,
    rng: Optional[np.random.Generator] = None,
    normalizevector: Optional[np.ndarray] = None,
    trace: Optional[Callable[[int, np.ndarray, np.ndarray, Optional[float]], None]] = None,
    info: Optional[dict] = None,
):
    """`NMFmultiplicative(X::AbstractMatrix, k)` src/NMFkMultiplicative.jl:24-127.

    Mutates X during the run (lambda substitution, NaN imputation) and restores it before
    returning, exactly like the reference.  `rng` stands in for Julia's global RNG
    (draw order W then H, :38,:48).  `trace(iter, W, H, obj_or_None)` is called at the end of
    the body of every iteration (so on the every-10th check iterations W,H carry the clamp of
    :99-100 and obj is the value of :74; obj is None otherwise) - used for per-iteration parity.
    Returns (W, H, objvalue) with objvalue the sum of squares of :125.
    """
    inan, izero = nmf_preprocessing(X, lam)  # :25
    n, m = X.shape
    weight = _julia_weight(weight, n, m)
    if normalizevector is not None and len(normalizevector) == n:  # :27-31
        X /= np.asarray(normalizevector).reshape(n, 1)
    elif normalizevector is not None and len(normalizevector) != 0:
        raise ValueError("Length of normalizing vector does not match")
    if rng is None:
        rng = np.random.default_rng()
    if Winit is None or Winit.size == 0:  # :37-45
        W = rng.random(n * k).reshape((n, k), order="F")
    else:
        assert Winit.shape == (n, k)
        W = Winit
        if np.isnan(W).any():
            raise ValueError("Initial values for the W matrix entries include NaNs!")
    if Hinit is None or Hinit.size == 0:  # :47-55
        H = rng.random(k * m).reshape((k, m), order="F")
    else:
        assert Hinit.shape == (k, m)
        H = Hinit
        if np.isnan(H).any():
            raise ValueError("Initial values for the H matrix entries include NaNs!")

    consold = None  # falses(m, m): never equals a real `cons` (its diagonal is true) when m > 0
    inc = 0
    objvalue_best = np.inf
    iters = 0
    baditers = 0
    reattempts = 0
    stop_reason = "maxiter"
    any_nan = bool(inan.any())
    while iters < maxiter and baditers < maxbaditers and reattempts < maxreattempts:  # :64
        iters += 1
        if not Hfixed:  # :66-68
            H = H * (W.T @ (X / (W @ H))) / np.sum(W, axis=0).reshape(k, 1)
        if not Wfixed:  # :69-71
            W = W * ((X / (W @ H)) @ H.T) / np.sum(H, axis=1).reshape(1, k)
        WH = W @ H  # the reference forms W*H again for the imputation, :72
        if any_nan:
            X[inan] = WH[inan]
        objvalue = None
        if iters % 10 == 0:  # :73
            objvalue = float(np.sum((((X - W @ H) * weight)[~inan]) ** 2))  # :74
            if objvalue < tol:  # :75-78
                stop_reason = "tol"
                if trace is not None:
                    trace(iters, W, H, objvalue)
                break
            if objvalue < objvalue_best:  # :79-88
                if (objvalue_best - objvalue) < tolOF:
                    baditers += 1
                else:
                    baditers = 0
                objvalue_best = objvalue
            else:
                baditers += 1
            if baditers >= maxbaditers:  # :90-98
                reattempts += 1
                baditers = 0
            H = np.maximum(H, EPS64)  # :99
            W = np.maximum(W, EPS64)  # :100
            index = np.argmin(H, axis=0)  # :101-103 (first minimum, like Julia argmin)
            cons = _canon_partition(index)  # :105
            if consold is not None and np.array_equal(cons, consold):  # :106-111
                inc += 1
            else:
                inc = 0
            if inc > stopconv:  # :112-115
                stop_reason = "consistency"
                if trace is not None:
                    trace(iters, W, H, objvalue)
                break
            consold = cons  # :116
        if trace is not None:
            trace(iters, W, H, objvalue)
    else:
        if iters >= maxiter:
            stop_reason = "maxiter"
        elif reattempts >= maxreattempts:
            stop_reason = "reattempts"
        else:
            stop_reason = "baditers"
    if normalizevector is not None and len(normalizevector) == n:  # :119-122
        nv = np.asarray(normalizevector).reshape(n, 1)
        X *= nv
        W = W * nv
    X[izero] = 0  # :123
    X[inan] = np.nan  # :124
    objvalue = float(np.sum((((X - W @ H) * weight)[~inan]) ** 2))  # :125
    if info is not None:
        info.update(iters=iters, stop_reason=stop_reason, baditers=baditers, reattempts=reattempts)
    return W, H, objvalue


def nmf_multiplicative_darray(
    X: np.ndarray,
    k: int,
    *,
    tol: float = 1e-19,
    lam: float = 1e-32,
    maxiter: int = 1000000,
    stopconv: int = 10000,
    Winit: Optional[np.ndarray] = None,
    Hinit: Optional[np.ndarray] = None,
    rng: Optional[np.random.Generator] = None,
    info: Optional[dict] = None,
):
    """`NMFmultiplicative(X::DArray, k)` src/NMFkMultiplicative.jl:129-197: the same two updates on distributed arrays, but NO
    tolOF / baditers / reattempts logic, no weight, no NaN imputation; the loop ends on objvalue < tol (:170-173), on
    inc > stopconv (default 10000, :186-189) or after maxiter iterations.  The distribution itself (collect / distribute of
    the k-vectors and of H', :160-167) does not change the arithmetic, so this is a dense restatement."""
    inan, izero = nmf_preprocessing(X, lam)  # :130
    n, m = X.shape
    if rng is None:
        rng = np.random.default_rng()
    W = rng.random(n * k).reshape((n, k), order="F") if Winit is None or Winit.size == 0 else Winit  # :136-144
    H = rng.random(k * m).reshape((k, m), order="F") if Hinit is None or Hinit.size == 0 else Hinit  # :146-154
    if np.isnan(W).any():
        raise ValueError("Initial values for the W matrix entries include NaNs!")
    if np.isnan(H).any():
        raise ValueError("Initial values for the H matrix entries include NaNs!")
    consold, inc, iters, stop_reason = None, 0, 0, "maxiter"
    for i in range(1, maxiter + 1):  # :159
        iters = i
        H = H * (W.T @ (X / (W @ H))) / np.sum(W, axis=0).reshape(k, 1)  # :160-162
        W = W * ((X / (W @ H)) @ H.T) / np.sum(H, axis=1).reshape(1, k)  # :163-167
        if i % 10 == 0:  # :168
            objvalue = float(np.sum((X - W @ H) ** 2))  # :169
            if objvalue < tol:  # :170-173
                stop_reason = "tol"
                break
            H = np.maximum(H, EPS64)  # :174
            W = np.maximum(W, EPS64)  # :175
            cons = _canon_partition(np.argmin(H, axis=0))  # :176-179
            inc = inc + 1 if (consold is not None and np.array_equal(cons, consold)) else 0  # :180-185
            if inc > stopconv:  # :186-189
                stop_reason = "consistency"
                break
            consold = cons  # :190
    X[izero] = 0  # :193
    X[inan] = np.nan  # :194
    objvalue = float(np.sum((X - W @ H) ** 2))  # :195
    if info is not None:
        info.update(iters=iters, stop_reason=stop_reason)
    return W, H, objvalue


# --------------------------------------------------------------------------------------
# Variant FRO: method=:nmf, algorithm=:multdiv (src/NMFkExecute.jl:763-766) -> NMF.MultUpdate(obj=:mse)
# --------------------------------------------------------------------------------------
def nmf_multupdate_mse(
    X: np.ndarray,
    k: int,
    *,
    Winit: np.ndarray,
    Hinit: np.ndarray,
    maxiter: int = 10000,
    tol: float = 1e-19,
    lambda_w: float = 0.0,
    lambda_h: float = 0.0,
    delta: Optional[float] = None,
    trace: Optional[Callable[[int, np.ndarray, np.ndarray], None]] = None,
    info: Optional[dict] = None,
):
    """The Frobenius ("mse") multiplicative update of the third-party package NMF.jl (compat "0.4-1", Project.toml:85; NOT
    vendored under /root/reference - restated from the published source `src/multupd.jl` + `src/common.jl`, unpinned), which
    the reference reaches at src/NMFkExecute.jl:763-766 (`NMF.solve!(NMF.MultUpdate{T}(obj=:mse, maxiter, tol), X, W, H)`; the
    reference's keyword for it is algorithm=:multdiv).  It is the update BASELINE.json's north star writes out:
        H <- H .* (W'X)  ./ (W'W*H  + lambda_h + delta)        delta = sqrt(eps(T))
        W <- W .* (X*H') ./ (W*H*H' + lambda_w + delta)        (with the new H)
    until every column of W and every row of H moved by less than `tol` relative (NMF.jl `stop_condition`:
    sqrt(sum((new-old)^2)) <= tol * sqrt(sum((new+old)^2)) for all of them) or `maxiter` iterations.  In the reference the
    initial factors come from NMF.randinit; here they are injected.  Computes in the dtype of the inputs (pass Float64 copies
    for a Float64 oracle of Float32 data; `delta` then still has to be sqrt(eps(Float32)), hence the argument).
    Returns (W, H, objvalue = sum((X - W*H)^2), the package's `sqL2dist`)."""
    W = np.array(Winit, copy=True)
    H = np.array(Hinit, copy=True)
    if delta is None:
        delta = float(np.sqrt(np.finfo(X.dtype).eps))
    iters, converged = 0, False
    while not converged and iters < maxiter:
        iters += 1
        preW, preH = W.copy(), H.copy()
        WtX = W.T @ X
        WtWH = (W.T @ W) @ H
        H *= WtX / (WtWH + (lambda_h + delta))
        XHt = X @ H.T
        WHHt = W @ (H @ H.T)
        W *= XHt / (WHHt + (lambda_w + delta))
        dw = np.sqrt(np.sum((W - preW) ** 2, axis=0))
        sw = np.sqrt(np.sum((W + preW) ** 2, axis=0))
        dh = np.sqrt(np.sum((H - preH) ** 2, axis=1))
        sh = np.sqrt(np.sum((H + preH) ** 2, axis=1))
        converged = not (np.any(dw > tol * sw) or np.any(dh > tol * sh))
        if trace is not None:
            trace(iters, W, H)
    if info is not None:
        info.update(iters=iters, converged=converged, stop_reason="tol" if converged else "maxiter")
    return W, H, float(np.sum((X - W @ H) ** 2))


def execute_singlerun_nmf(X: np.ndarray, nk: int, *, Winit, Hinit, maxiter: int = 10000, tol: float = 1e-19,
                          modifymatrices: bool = True, info: Optional[dict] = None, delta: Optional[float] = None):
    """`execute_singlerun_compute(X, nk; method=:nmf, algorithm=:multdiv)` src/NMFkExecute.jl:763-775, 787-805: the solver
    above, then objvalue = normnan(X - W*H) and the H-row normalisation like every other method."""
    W, H, _ = nmf_multupdate_mse(X, nk, Winit=Winit, Hinit=Hinit, maxiter=maxiter, tol=tol, delta=delta, info=info)
    objvalue = normnan(X - W @ H)
    if modifymatrices:
        total = np.sum(H, axis=1, keepdims=True)
        W = W * total.T
        H = H / total
    return W, H, objvalue


# --------------------------------------------------------------------------------------
# NMFsparsity: src/NMFkSparsity.jl:1-113 (method=:sparsity, src/NMFkExecute.jl:757-758)
# --------------------------------------------------------------------------------------
def nmf_sparsity(X: np.ndarray, k: int, *, cost_function: str = "ed", beta_divergence: float = -1, sparsity: float = 1,
                 maxiter: int = 100000, tol: float = 1e-19, lam: float = 1e-9, Winit: Optional[np.ndarray] = None,
                 Hinit: Optional[np.ndarray] = None, rng: Optional[np.random.Generator] = None, info: Optional[dict] = None,
                 trace: Optional[Callable[[int, np.ndarray, np.ndarray, float], None]] = None):
    """`NMFsparsity(X, k; cost_function=:ed, beta_divergence=-1, sparsity=1, maxiter, tol, lambda=1e-9, Winit, Hinit)`
    src/NMFkSparsity.jl:1-113 with w_ind = h_ind = trues(k): beta-divergence multiplicative updates with an L1 penalty on H
    and unit-norm columns of W.  X_est = max.(W*H, lambda) is re-formed after every half-update (:71, :88); the run stops when
    the relative change of (divergence + sparsity * sum(H)) drops below tol (:101-106).  Returns (W, H, sum((X - W*H)^2))."""
    if beta_divergence == -1:  # :5-22
        beta_divergence = {"kl": 1, "ed": 2, "is": 0}.get(cost_function, 2)
    b = beta_divergence
    n, m = X.shape
    if rng is None:
        rng = np.random.default_rng()
    W = rng.random(n * k).reshape((n, k), order="F") if Winit is None or Winit.size == 0 else np.array(Winit, copy=True)  # :31-36
    H = rng.random(k * m).reshape((k, m), order="F") if Hinit is None or Hinit.size == 0 else np.array(Hinit, copy=True)  # :37-42
    Wn = np.sqrt(np.sum(W ** 2, axis=0, keepdims=True))  # :44-46
    W = W / Wn
    H = H * Wn.T
    X_est = np.maximum(W @ H, lam)  # :48
    it, last_of, of, stop = 0, None, None, "maxiter"
    while it < maxiter:  # :56
        it += 1
        if b == 1:  # :59-61
            dph = np.sum(W, axis=0).reshape(k, 1) + sparsity
            dmh = W.T @ (X / X_est)
        elif b == 2:  # :62-64
            dph = W.T @ X_est + sparsity
            dmh = W.T @ X
        else:  # :65-67
            dph = W.T @ X_est ** (b - 1) + sparsity
            dmh = W.T @ (X * X_est ** (b - 2))
        dph = np.maximum(dph, lam)  # :69
        H = H * (dmh / dph)  # :70
        X_est = np.maximum(W @ H, lam)  # :71
        if b == 1:  # :74-76
            A = (X / X_est) @ H.T
            dpw = np.sum(H, axis=1).reshape(1, k) + np.sum(A * W, axis=0, keepdims=True) * W
            dmw = A + np.sum(np.sum(H, axis=1).reshape(1, k) * W, axis=0, keepdims=True) * W
        elif b == 2:  # :77-79
            dpw = X_est @ H.T + np.sum((X @ H.T) * W, axis=0, keepdims=True) * W
            dmw = X @ H.T + np.sum((X_est @ H.T) * W, axis=0, keepdims=True) * W
        else:  # :80-82
            A1, A2 = X_est ** (b - 1) @ H.T, (X * X_est ** (b - 2)) @ H.T
            dpw = A1 + np.sum(A2 * W, axis=0, keepdims=True) * W
            dmw = A2 + np.sum(A1 * W, axis=0, keepdims=True) * W
        dpw = np.maximum(dpw, lam)  # :84
        W = W * (dmw / dpw)  # :85
        W = W / np.sqrt(np.sum(W ** 2, axis=0, keepdims=True))  # :86
        X_est = np.maximum(W @ H, lam)  # :87
        if b == 1:  # :89-98
            div = float(np.sum(X * np.log(X / X_est) - X + X_est))
        elif b == 2:
            div = float(np.sum((X - X_est) ** 2))
        elif b == 0:
            div = float(np.sum(X / X_est - np.log(X / X_est) - 1))
        else:
            div = float(np.sum(X ** b + (b - 1) * X_est ** b - b * X * X_est ** (b - 1)) / (b * (b - 1)))
        of = div + float(np.sum(H * sparsity))  # :99
        if trace is not None:
            trace(it, W, H, of)
        if it > 1 and tol > 0 and (abs(of - last_of) / last_of) < tol:  # :101-106
            stop = "tol"
            break
        last_of = of
    if info is not None:
        info.update(iters=it, stop_reason=stop, objective=of)
    return W, H, float(np.sum((X - W @ H) ** 2))  # :109-110


# --------------------------------------------------------------------------------------
# One restart as reached from execute: src/NMFkExecute.jl:729-807
# --------------------------------------------------------------------------------------
def execute_singlerun_compute(
    X: np.ndarray,
    nk: int,
    *,
    maxiter: int = 10000,
    tol: float = 1e-19,
    clusterWmatrix: bool = False,
    modifymatrices: bool = True,
    weight=1,
    method: str = "simple",
    info: Optional[dict] = None,
    **kw,
):
    """`execute_singlerun_compute(X::AbstractMatrix, nk; method=:simple, ...)`
    src/NMFkExecute.jl:729-807 with scale=false, transpose=false, mixture=:null.
    X is passed by reference (:740) and comes back restored.  Returns (W, H, objvalue) where
    objvalue = normnan(X - W*H) (:791-792, a NORM) and rows of H sum to one (:800-804).
    method="sparsity" solves with NMFsparsity(X, nk; maxiter, tol, kw...) (:757-758) instead: kw takes cost_function,
    beta_divergence, sparsity and lam (its `lambda`); the weight does not reach it."""
    if method == "sparsity":
        W, H, _ = nmf_sparsity(X, nk, maxiter=maxiter, tol=tol, info=info, **kw)  # :757-758
    elif method == "simple":
        W, H, _ = nmf_multiplicative(X, nk, tol=tol, maxiter=maxiter, weight=weight, info=info, **kw)  # :762
    else:
        raise ValueError("method=:%s is not restated here (:simple and :sparsity are)" % method)
    E = X - W @ H  # :791
    objvalue = normnan(E)  # :792
    if modifymatrices:  # :795-805 (mixture == :null)
        if clusterWmatrix:
            total = np.sum(W, axis=0, keepdims=True)
            W = W / total
            H = H * total.T
        else:
            total = np.sum(H, axis=1, keepdims=True)
            W = W * total.T
            H = H / total
    return W, H, objvalue


# --------------------------------------------------------------------------------------
# Third-party semantics (Distances.jl, Clustering.jl), restated
# --------------------------------------------------------------------------------------
def cosine_dist(a: np.ndarray, b: np.ndarray) -> float:
    """Distances.cosine_dist(a,b) = max(1 - a.b / (sqrt(a.a) * sqrt(b.b)), 0)
    (Distances.jl `CosineDist` eval_reduce/eval_end), call site src/NMFkCluster.jl:470."""
    ab = float(np.dot(a, b))
    a2 = float(np.dot(a, a))
    b2 = float(np.dot(b, b))
    with np.errstate(divide="ignore", invalid="ignore"):
        v = np.float64(1.0) - np.float64(ab) / (np.sqrt(np.float64(a2)) * np.sqrt(np.float64(b2)))
    if math.isnan(v):
        return float("nan")
    return float(max(v, 0.0))


def pairwise_cosine_rows(V: np.ndarray) -> np.ndarray:
    """Distances.pairwise(CosineDist(), V; dims=1) (Distances.jl `_pairwise!(r, ::CosineDist, a)`):
    Gram matrix by BLAS, r[i,j] = max(1 - G[i,j]/(sqrt(G[i,i])*sqrt(G[j,j])), 0), diagonal forced
    to 0, symmetric.  Call site src/NMFkFinalize.jl:52."""
    G = V @ V.T
    nrm = np.sqrt(np.diag(G))
    with np.errstate(divide="ignore", invalid="ignore"):
        D = 1.0 - G / (nrm[:, None] * nrm[None, :])
    D = np.where(np.isnan(D), D, np.maximum(D, 0.0))
    # lower triangle is computed, upper is its mirror, diagonal is exactly zero
    iu = np.triu_indices(V.shape[0], 1)
    D[iu] = D.T[iu]
    np.fill_diagonal(D, 0.0)
    return D


def silhouettes(assignments: np.ndarray, dists: np.ndarray) -> np.ndarray:
    """Clustering.silhouettes(assignments, dists) (Clustering.jl 0.14/0.15 `silhouettes.jl`):
    r[c,j] = sum_{i != j, a_i = c} dists[i,j]; divided by counts[c] - (c == a_j) (0 if that
    is 0); a = r[a_j,j]; b = min_{c != a_j} r[c,j]; s = a<b ? 1-a/b : a>b ? b/a-1 : 0;
    s = 0 for singleton clusters.  assignments are 1-based.  Call site NMFkFinalize.jl:55."""
    a_ = np.asarray(assignments, dtype=np.int64) - 1
    n = len(a_)
    k = int(a_.max()) + 1
    if k < 2:
        raise ValueError("silhouettes() not defined for the degenerated clustering with a single cluster.")
    counts = np.bincount(a_, minlength=k)
    onehot = np.zeros((k, n), dtype=dists.dtype)
    onehot[a_, np.arange(n)] = 1
    D = np.array(dists, copy=True)
    np.fill_diagonal(D, 0.0)  # the i == j term is skipped
    r = onehot @ D  # r[c, j]
    for j in range(n):
        for c in range(k):
            cnt = counts[c] - (1 if c == a_[j] else 0)
            r[c, j] = 0.0 if cnt == 0 else r[c, j] / cnt
    sil = np.zeros(n, dtype=r.dtype)
    for j in range(n):
        l = a_[j]
        a = r[l, j]
        others = np.delete(r[:, j], l)
        # typemax start + strict '<' scan == plain minimum (NaN never wins a '<')
        b = np.inf
        for v in others:
            if v < b:
                b = v
        if counts[l] == 1:
            sil[j] = 0
        else:
            sil[j] = (1 - a / b) if a < b else ((b / a - 1) if a > b else 0.0)
    return sil


# --------------------------------------------------------------------------------------
# Solution clustering: src/NMFkCluster.jl:425-517
# --------------------------------------------------------------------------------------
def clustersolutions(factors: Sequence[np.ndarray], clusterWmatrix: bool = False):
    """`clustersolutions(factors, clusterWmatrix=false)` src/NMFkCluster.jl:425-517.
    Returns (labels k x R, 1-based; centroids)."""
    if not clusterWmatrix:
        factors = [np.array(f.T, copy=True) for f in factors]  # :427 permutedims makes copies
    else:
        # NO copy on this branch (:426-428): factors[1] below IS the caller's best W, which the running-sum
        # centroids then overwrite in place (:453-455, :484, :512) - execute_run reads it afterwards (:631-637)
        factors = list(factors)
    numTrials = len(factors)
    r, k = factors[0].shape
    for w in factors:
        assert w.shape == (r, k)
    needZeroFix = any(np.min(np.sum(f, axis=0)) == 0 for f in factors)  # :437-444
    if needZeroFix:  # :445-450
        factors = [np.vstack([f, np.ones((1, k), dtype=f.dtype)]) for f in factors]
    cent = factors[0]  # centSeeds and newClusterCenters alias factors[1], :453-455
    labels = np.zeros((k, numTrials), dtype=np.int64)
    labels[:, 0] = np.arange(1, k + 1)  # :461
    D = np.empty((k, k), dtype=factors[0].dtype)
    for trial in range(1, numTrials):  # :464
        Wt = factors[trial]
        for c in range(k):  # :467-472
            centroid = cent[:, c].copy()
            for f in range(k):
                D[f, c] = cosine_dist(Wt[:, f], centroid)
        D[np.isnan(D)] = 0  # :473
        while np.min(D) < np.inf:  # :474-485
            flat = int(np.argmin(D.T))  # column-major first minimum
            c, f = divmod(flat, k)
            labels[f, trial] = c + 1
            D[f, :] += np.inf
            D[:, c] += np.inf
            cent[:, c] += Wt[:, f]
    while labels.min() == 0:  # :487-496
        flat = int(np.argmin(labels.T))
        trial, idx = divmod(flat, k)
        if labels[:, trial].sum() == 0:
            labels[:, trial] = np.arange(1, k + 1)
        else:
            labels[idx, trial] = idx + 1
    cent /= numTrials  # :512 `newClusterCenters ./= numTrials` (in place: the aliased best W ends up holding the centroids)
    return labels, cent.T.copy()  # :516


# --------------------------------------------------------------------------------------
# robustkmeans: src/NMFkCluster.jl:138-289 (+ Clustering.jl `kmeans`, restated)
# --------------------------------------------------------------------------------------
def pairwise_cosine_cols(A: np.ndarray, B: np.ndarray) -> np.ndarray:
    """Distances.pairwise(CosineDist(), A, B; dims=2): r[i,j] = max(1 - <A[:,i],B[:,j]> / (|A[:,i]| |B[:,j]|), 0)."""
    G = A.T @ B
    ra = np.sqrt(np.sum(A * A, axis=0))
    rb = np.sqrt(np.sum(B * B, axis=0))
    with np.errstate(divide="ignore", invalid="ignore"):
        D = 1.0 - G / (ra[:, None] * rb[None, :])
    return np.where(np.isnan(D), D, np.maximum(D, 0.0))


def kmeans_lloyd(X: np.ndarray, k: int, seeds: Sequence[int], maxiter: int = 1000, tol: float = 1e-32):
    """Clustering.kmeans(X, k; maxiter, tol, distance=CosineDist()) from given seeds (Clustering.jl 0.14/0.15 `kmeans.jl`
    `_kmeans!`, `update_assignments!`, `update_centers!`, restated; the package is not vendored under /root/reference).  The points
    are the COLUMNS of X (d x N).  The package draws the seeds with k-means++ from Julia's RNG (not reproducible here: an input)
    and re-draws a centre that lost all its points at random (`repick_unused_centers`; here such a centre keeps its position,
    and `empty` reports that it happened).  Returns a dict with the fields of KmeansResult."""
    d, n = X.shape
    centers = np.array(X[:, list(seeds)], dtype=np.float64, copy=True)
    assignments = np.zeros(n, dtype=np.int64)
    costs = np.zeros(n)
    counts = np.zeros(k, dtype=np.int64)
    to_update = np.ones(k, dtype=bool)

    def update_assignments(dmat, is_init):
        nonlocal to_update
        to_update[:] = is_init
        counts[:] = 0
        for j in range(n):
            c, a = 0, dmat[0, j]
            for i in range(1, k):
                if dmat[i, j] < a:
                    a, c = dmat[i, j], i
            if is_init:
                assignments[j] = c
            elif c != assignments[j]:
                to_update[c] = True
                to_update[assignments[j]] = True
                assignments[j] = c
            costs[j] = a
            counts[c] += 1
        unused = [i for i in range(k) if counts[i] == 0]
        for i in unused:
            to_update[i] = False
        return unused

    unused = update_assignments(pairwise_cosine_cols(centers, X), True)
    objv = float(np.sum(costs))
    t, converged, empty = 0, False, False
    while not converged and t < maxiter:
        t += 1
        for c in range(k):  # update_centers!: mean of the assigned points for the clusters whose membership changed
            if to_update[c] and counts[c] > 0:
                centers[:, c] = X[:, assignments == c].sum(axis=1) / counts[c]
        empty = empty or bool(unused)
        unused = update_assignments(pairwise_cosine_cols(centers, X), False)
        prev, objv = objv, float(np.sum(costs))
        change = objv - prev
        if change > tol:
            pass  # "The clustering cost increased at iteration"
        elif k == 1 or abs(change) < tol:
            converged = True
    return dict(centers=centers, assignments=assignments + 1, costs=costs.copy(), counts=counts.copy(), totalcost=objv, iterations=t,
                converged=converged, empty=empty)


def sortclustering(res: dict) -> dict:
    """`sortclustering(c::Clustering.KmeansResult)` src/NMFkCluster.jl:264-289: relabel the clusters in order of first appearance,
    then rank them by size (descending, stable)."""
    a = res["assignments"]
    j = list(dict.fromkeys(a.tolist()))  # unique, order of first appearance
    relabel = {lab: q + 1 for q, lab in enumerate(j)}
    ca = np.array([relabel[v] for v in a])
    cnt = np.array([res["counts"][lab - 1] for lab in j])
    i = np.argsort(-cnt, kind="stable")
    ca2 = np.zeros_like(ca)
    for q, idx in enumerate(i):
        ca2[ca == idx + 1] = q + 1
    r = [j[idx] - 1 for idx in i]
    out = dict(res)
    out.update(assignments=ca2, centers=res["centers"][:, r], counts=res["counts"][r])
    return out


def robustkmeans(X: np.ndarray, k: int, seeds_per_repeat: Sequence[Sequence[int]], maxiter: int = 1000, tol: float = 1e-32,
                 compute_silhouettes_flag: bool = False):
    """`robustkmeans(X, k, repeats; ...)` src/NMFkCluster.jl:172-246 with the seeds of every repeat injected: the first repeat
    with the smallest total cost wins (:219-225), silhouettes on pairwise(CosineDist(), zerostoepsilon(X); dims=2) (:195-214),
    then sortclustering (:227).  Returns (result dict, best_silhouettes or None)."""
    best, best_cost, best_sil = None, np.inf, np.zeros(X.shape[1])
    Xd = pairwise_cosine_rows(zerostoepsilon(X).T) if compute_silhouettes_flag else None
    for i, seeds in enumerate(seeds_per_repeat):
        c = kmeans_lloyd(X, k, seeds, maxiter, tol)
        if i == 0 or c["totalcost"] < best_cost:
            best, best_cost = c, c["totalcost"]
            if compute_silhouettes_flag:
                best_sil = silhouettes(c["assignments"], Xd) if c["assignments"].max() > 1 else np.zeros(X.shape[1])
    return sortclustering(best), (best_sil if compute_silhouettes_flag else None)


# --------------------------------------------------------------------------------------
# finalize: src/NMFkFinalize.jl:36-79
# --------------------------------------------------------------------------------------
def finalize(Wa: Sequence[np.ndarray], Ha: Sequence[np.ndarray], idx: np.ndarray, clusterWmatrix: bool = False):
    """`finalize(Wa::Vector, Ha::Vector, idx::Matrix, clusterWmatrix=false)`
    src/NMFkFinalize.jl:36-79.  Returns (W, H, clustersilhouettes, Wvar, Hvar)."""
    nNMF = len(Wa)
    nP = Wa[0].shape[0]
    nk, nC = Ha[0].shape
    idx_r = idx.reshape(-1, order="F")  # :43
    if clusterWmatrix:
        V = zerostoepsilon(np.hstack(Wa)).T  # pairwise over columns == rows of the transpose
    else:
        V = zerostoepsilon(np.vstack(Ha))  # :52
    Dm = pairwise_cosine_rows(V)
    Dm[np.isnan(Dm)] = 0  # :53-54
    sil = silhouettes(idx_r, Dm).reshape((nk, nNMF), order="F")  # :55
    sil[np.isnan(sil)] = 0  # :58
    dt = Ha[0].dtype
    clustersil = np.empty((nk, 1), dtype=dt)
    W = np.empty((nP, nk), dtype=dt)
    H = np.empty((nk, nC), dtype=dt)
    Wvar = np.empty((nP, nk), dtype=dt)
    Hvar = np.empty((nk, nC), dtype=dt)
    for c in range(1, nk + 1):  # :64-77
        mask = idx == c
        clustersil[c - 1, 0] = np.mean(sil.T[mask.T])  # column-major order of findall
        # idxkk: for every (row a, trial t) with idx[a,t] == c, in column-major order, the row a
        cm = [(a, t) for t in range(nNMF) for a in range(nk) if idx[a, t] == c]
        idxkk = [a for a, _ in cm]
        # map((i, j)->Wa[i][:, j], 1:nNMF, idxkk) zips trial i with the i-th hit's row
        ws = np.stack([Wa[i][:, j] for i, j in zip(range(nNMF), idxkk)], axis=1)
        hs = np.stack([Ha[i][j, :] for i, j in zip(range(nNMF), idxkk)], axis=1)
        H[c - 1, :] = hs.mean(axis=1)
        W[:, c - 1] = ws.mean(axis=1)
        Wvar[:, c - 1] = ws.var(axis=1, ddof=1) if ws.shape[1] > 1 else np.nan
        Hvar[c - 1, :] = hs.var(axis=1, ddof=1) if hs.shape[1] > 1 else np.nan
    return W, H, clustersil, Wvar, Hvar


# --------------------------------------------------------------------------------------
# k selection and ordering: src/NMFkPostprocess.jl:7-41, 148-158
# --------------------------------------------------------------------------------------
def getk(nkrange: Sequence[int], robustness: Sequence[float], cutoff: float = 0.5, strict: bool = True):
    """`getk` src/NMFkPostprocess.jl:7-41.  `robustness` has one entry per element of nkrange
    (the caller indexes `robustness[nkrange]`, NMFkExecute.jl:225).  Returns k, 0 or None."""
    nkrange = list(nkrange)
    robustness = np.asarray(robustness, dtype=float)
    if len(nkrange) != len(robustness):  # :8-10
        robustness = robustness[np.asarray(nkrange) - 1]
    if np.all(np.isnan(robustness)):  # :11-13
        return 0
    if len(nkrange) == 1:  # :14-23
        if strict:
            return nkrange[-1] if robustness[-1] > cutoff else None
        return nkrange[-1]
    hits = np.flatnonzero(robustness > cutoff)  # :25
    if len(hits) == 0:
        if strict:
            return None
        rb = np.where(np.isnan(robustness), -np.inf, robustness)
        return nkrange[int(np.argmax(rb))]
    return nkrange[int(hits[-1])]


def signalorder(W: np.ndarray, H: np.ndarray) -> np.ndarray:
    """`signalorder` src/NMFkPostprocess.jl:148-158 : sortperm(sum(W[:,i]*H[i,:]); rev=true).
    Returns 0-based indices."""
    k = W.shape[1]
    assert k == H.shape[0]
    s = np.array([np.sum(np.outer(W[:, i], H[i, :])) for i in range(k)])
    return np.argsort(-s, kind="stable")


# --------------------------------------------------------------------------------------
# execute_run / execute: src/NMFkExecute.jl:483-711, 178-329
# --------------------------------------------------------------------------------------
def execute_run(
    X: np.ndarray,
    nk: int,
    nNMF: int,
    *,
    clusterWmatrix: bool = False,
    weight=1,
    seed: Optional[int] = None,
    inits: Optional[Sequence] = None,
    init_fn: Optional[Callable[[int, int, int, int], tuple]] = None,
    details: Optional[dict] = None,
    best: bool = True,
    acceptratio: float = 1,
    acceptfactor: float = np.inf,
    nanaction: str = "zeroed",
    **kw,
):
    """`execute_run(X::AbstractMatrix, nk, nNMF; ...)` src/NMFkExecute.jl:483-711 (serial branch); best=false returns
    the per-cluster means of finalize (:637, :655-658) instead of the best restart; acceptratio / acceptfactor /
    nanaction filter the solutions that reach clustersolutions / finalize (:551-597).

    Initialisations: the reference draws from Julia's RNG (seed+i per restart when `seed` is
    given, :532-537).  Here `inits[i] = (Winit, Hinit)` or `init_fn(i, n, nk, m)` (i is the
    1-based restart number) supply them explicitly (SURVEY.md §8c: inject Winit/Hinit).
    Returns (Wa, Ha, phi, minsilhouette, aic)."""
    T = X.dtype
    n, m = X.shape
    modifymatrices = not ("Wfixed" in kw or "Hfixed" in kw)  # :486-489
    WBig, HBig, objvalue, iters, stops = [], [], np.empty(nNMF, dtype=T), [], []
    for i in range(1, nNMF + 1):  # :534-542
        kwi = dict(kw)
        if inits is not None:
            kwi["Winit"], kwi["Hinit"] = inits[i - 1]
        elif init_fn is not None:
            kwi["Winit"], kwi["Hinit"] = init_fn(i, n, nk, m)
        elif seed is not None:
            kwi["rng"] = np.random.Generator(np.random.Philox(key=seed + i))
        inf = {}
        # clusterWmatrix is a named keyword of execute_run and is NOT forwarded (:516-540): every restart is normalised
        # with the default branch (rows of H sum to one, :800-804)
        W, H, of = execute_singlerun_compute(X, nk, modifymatrices=modifymatrices, weight=weight, info=inf, **kwi)
        WBig.append(np.array(W, dtype=T))  # stored into Vector{Matrix{T}}, :529-536
        HBig.append(np.array(H, dtype=T))
        objvalue[i - 1] = of
        iters.append(inf.get("iters", 0))
        stops.append(inf.get("stop_reason", ""))
    idxsort = np.argsort(objvalue, kind="stable")  # :545 sortperm
    bestIdx = int(idxsort[0])
    Wbest = WBig[bestIdx].copy()  # :549-550
    Hbest = HBig[bestIdx].copy()
    if acceptratio < 1:  # :552-558
        ccc = int(math.ceil(nNMF * acceptratio))
        idxrat = np.array([True] * ccc + [False] * (nNMF - ccc))
    else:
        idxrat = np.ones(nNMF, dtype=bool)
    if acceptfactor < np.inf:  # :559-565
        idxcut = objvalue[idxsort] < objvalue[bestIdx] * acceptfactor
    else:
        idxcut = np.ones(nNMF, dtype=bool)
    idxnan = np.ones(nNMF, dtype=bool)
    if nanaction == "zeroed":  # :566-580
        for i in idxsort:
            WBig[i][np.isnan(WBig[i])] = 0
            HBig[i][np.isnan(HBig[i])] = 0
    elif nanaction == "removed":  # :581-596 (idxnan is indexed by restart NUMBER, the other two by sorted position)
        for i in idxsort:
            if np.isnan(WBig[i]).any() or np.isnan(HBig[i]).any():
                idxnan[i] = False
    idxsol = idxrat & idxcut & idxnan  # :597
    minsilhouette = 1
    labels = None
    clustersil = None
    centroids = None
    Wv = Hv = np.nan
    Ws = [WBig[i] for i in idxsort[idxsol]]  # WBig[idxsort][idxsol]
    Hs = [HBig[i] for i in idxsort[idxsol]]
    if nk > 1:  # :618-645
        labels, centroids = clustersolutions(Ws if clusterWmatrix else Hs, clusterWmatrix)  # :620-624
        ci = labels[:, 0]
        for i, c in enumerate(ci):  # :631-635 (reads WBig[bestIdx] AFTER clustersolutions may have overwritten it)
            Wbest[:, i] = WBig[bestIdx][:, c - 1]
            Hbest[i, :] = HBig[bestIdx][c - 1, :]
        Wmean, Hmean, clustersil, Wv, Hv = finalize(Ws, Hs, labels, clusterWmatrix)  # :637
        minsilhouette = T.type(np.min(clustersil))  # :638
    else:  # :646-650: finalize(WBig[idxsol], HBig[idxsol]) -> mean over the single column / row of the FIRST kept restart
        keep = [i for i in range(nNMF) if idxsol[i]]
        Wmean = np.mean(WBig[keep[0]], axis=1, keepdims=True)
        Hmean = np.mean(HBig[keep[0]], axis=0, keepdims=True)
    Wa, Ha = (Wbest, Hbest) if best else (Wmean, Hmean)  # :655-658
    E = X - Wa @ Ha  # :664
    E[np.isnan(E)] = 0  # :667
    phi_final = normnan(E)  # :668
    numobservations = int(np.sum(~np.isnan(X)))  # :697
    numparameters = Wa.size + Ha.size  # :698
    with np.errstate(divide="ignore"):
        aic = 2 * numparameters + numobservations * math.log(phi_final / numobservations) if phi_final > 0 else -math.inf  # :708
    if details is not None:  # the fields of the "-all" result file (:650-654) and what the tests compare
        details.update(objvalue=objvalue, idxsort=idxsort, idxsol=idxsol, labels=labels, clustersil=clustersil,
                       centroids=centroids, iters=np.asarray(iters), stop_reasons=stops, WBig=WBig, HBig=HBig, Wmean=Wmean, Hmean=Hmean, Wvar=Wv,
                       Hvar=Hv, Wbest=Wbest, Hbest=Hbest)
    return Wa, Ha, T.type(phi_final), minsilhouette, aic


def execute_k(X, nk, nNMF=10, *, ordersignals=True, **kw):
    """`execute(X, nk::Integer, nNMF)` src/NMFkExecute.jl:236-329 without the file cache
    (load=false, save=false).  Returns (W[:,so], H[so,:], fit, robustness, aic)."""
    if X.size == 0:
        raise ValueError("Input array has a zero dimension!")  # :242-244
    if "Wfixed" in kw or "Hfixed" in kw:  # :305-307
        ordersignals = False
    W, H, fit, rob, aic = execute_run(X, nk, nNMF, **kw)  # :309
    so = signalorder(W, H) if ordersignals else np.arange(W.shape[1])  # :311-318
    return W[:, so], H[so, :], fit, rob, aic


def execute(X, nkrange, nNMF=10, *, cutoff=0.5, per_k_kw: Optional[Callable[[int], dict]] = None, **kw):
    """`execute(X, nkrange, nNMF; cutoff=0.5, ...)` src/NMFkExecute.jl:178-233 without file IO.
    Returns (W dict-by-k, H dict-by-k, fitquality[maxk], robustness[maxk], aic[maxk], kopt)."""
    nkrange = list(nkrange)
    T = X.dtype
    maxk = max(nkrange)
    W, H = {}, {}
    fitquality = np.zeros(maxk, dtype=T)
    robustness = np.zeros(maxk, dtype=T)
    aic = np.zeros(maxk, dtype=T)
    fitquality[0] = np.inf  # :200
    robustness[0] = -1  # :201
    for nk in nkrange:  # :203-205
        kwk = dict(kw)
        if per_k_kw is not None:
            kwk.update(per_k_kw(nk))
        W[nk], H[nk], fitquality[nk - 1], robustness[nk - 1], aic[nk - 1] = execute_k(X, nk, nNMF, **kwk)
    idx = np.asarray(nkrange) - 1
    if np.all(np.isinf(fitquality[idx])):  # :206-208
        kopt = 0
    else:
        for nk in nkrange:  # :211-222
            fitquality[nk - 1] = normnan(X - W[nk] @ H[nk])
        kopt = getk(nkrange, robustness[idx], cutoff)  # :225
    return W, H, fitquality, robustness, aic, kopt


# --------------------------------------------------------------------------------------
# Deterministic initialisations shared by the parity tests and the bench harness
# (SURVEY.md §8d: restart i uses Philox(key=seed0+i), draws W (column-major) then H)
# --------------------------------------------------------------------------------------
def philox_init(seed0: int, i: int, n: int, k: int, m: int, dtype=np.float64):
    rng = np.random.Generator(np.random.Philox(key=seed0 + i))
    W = rng.random(n * k).reshape((n, k), order="F").astype(dtype)
    H = rng.random(k * m).reshape((k, m), order="F").astype(dtype)
    return W, H
