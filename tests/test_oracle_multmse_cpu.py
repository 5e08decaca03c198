"""Reference restatement of NMF.jl's KL update (method=:nmf, algorithm=:multmse -> NMF.MultUpdate(obj=:div)), which
tests/test_gpu_multmse.py checks the device against, and its CPU tests: against the oracle's NMFmultiplicative
(oracle/nmfk_oracle.py) and a hand-checked stop rule.  No GPU.

The restatement lives here rather than in oracle/ so that the oracle the other variants are checked against stays as it is;
it follows the conventions of oracle/nmfk_oracle.py::nmf_multupdate_mse, its mse sibling."""
from typing import Callable, Optional

import numpy as np

from oracle import nmfk_oracle as o


def multupdate_div_delta(dtype) -> float:
    """delta of NMF.jl's MultUpdDiv: sqrt(eps(T)) - the same unpinned reading of NMF.jl as nmf_multupdate_mse's delta.  The one
    place the tests take it from."""
    return float(np.sqrt(np.finfo(dtype).eps))


def stop_condition(W, preW, H, preH, tol) -> bool:
    """NMF.jl `stop_condition`: every column of W and every row of H moved by at most `tol` relative (the criterion of
    nmf_multupdate_mse)."""
    dw = np.sqrt(np.sum((W - preW) ** 2, axis=0))
    sw = np.sqrt(np.sum((W + preW) ** 2, axis=0))
    dh = np.sqrt(np.sum((H - preH) ** 2, axis=1))
    sh = np.sqrt(np.sum((H + preH) ** 2, axis=1))
    return not (np.any(dw > tol * sw) or np.any(dh > tol * sh))


def nmf_multupdate_div(X: np.ndarray, k: int, *, Winit: np.ndarray, Hinit: np.ndarray, maxiter: int = 10000, tol: float = 1e-19,
                       delta: Optional[float] = None, trace: Optional[Callable[[int, np.ndarray, np.ndarray], None]] = None,
                       info: Optional[dict] = None):
    """The KL ("div") multiplicative update of the third-party package NMF.jl (not vendored by the reference - restated from
    the published source `src/multupd.jl` (`MultUpdDiv`, lambda_w = lambda_h = 0) + `src/common.jl`, unpinned, like
    nmf_multupdate_mse), which the reference reaches with method=:nmf, algorithm=:multmse (src/NMFkExecute.jl:765-768: the
    reference swaps the names, :multmse is `NMF.MultUpdate(obj=:div)`):
        Q = X ./ (W*H .+ delta);   H .*= (W'Q) ./ (colsum(W)' .+ delta)
        Q = X ./ (W*H .+ delta);   W .*= (Q*H') ./ (rowsum(H)' .+ delta)          (with the new H)
    delta = sqrt(eps(T)) (multupdate_div_delta), inside nmf_skeleton!'s loop `while !converged && t < maxiter` with
    stop_condition after every iteration.  X is used as given: zeros stay zeros, no lambda substitution, no clamp, no NaN
    handling.  Computes in the dtype of the inputs (pass Float64 copies and the `delta` of the data type for a Float64
    reference of Float32 data).  The products are written U * N / (sums + delta), the order of nmf_multiplicative, so that
    with delta = 0 and strictly positive X the two agree bit for bit until its first clamp.
    Returns (W, H, gkldiv(X, W*H) = sum(x log(x / wh) - x + wh), with 0 log 0 = 0)."""
    W = np.array(Winit, copy=True)
    H = np.array(Hinit, copy=True)
    if delta is None:
        delta = multupdate_div_delta(X.dtype)
    iters, converged = 0, False
    while not converged and iters < maxiter:
        iters += 1
        preW, preH = W.copy(), H.copy()
        H = H * (W.T @ (X / (W @ H + delta))) / (np.sum(W, axis=0).reshape(k, 1) + delta)
        W = W * ((X / (W @ H + delta)) @ H.T) / (np.sum(H, axis=1).reshape(1, k) + delta)
        converged = stop_condition(W, preW, H, preH, tol)
        if trace is not None:
            trace(iters, W, H)
    if info is not None:
        info.update(iters=iters, converged=converged, stop_reason="tol" if converged else "maxiter")
    WH = W @ H
    pos = X > 0
    gkl = float(np.sum(X[pos] * np.log(X[pos] / WH[pos])) - np.sum(X) + np.sum(WH))
    return W, H, gkl


def execute_singlerun_nmf_multmse(X: np.ndarray, nk: int, *, Winit, Hinit, maxiter: int = 10000, tol: float = 1e-19,
                                  modifymatrices: bool = True, info: Optional[dict] = None, delta: Optional[float] = None):
    """`execute_singlerun_compute(X, nk; method=:nmf, algorithm=:multmse)` src/NMFkExecute.jl:765-775, 787-805: the solver
    above, then objvalue = normnan(X - W*H) and the H-row normalisation like every other method."""
    W, H, _ = nmf_multupdate_div(X, nk, Winit=Winit, Hinit=Hinit, maxiter=maxiter, tol=tol, delta=delta, info=info)
    objvalue = o.normnan(X - W @ H)
    if modifymatrices:
        total = np.sum(H, axis=1, keepdims=True)
        W = W * total.T
        H = H / total
    return W, H, objvalue


def test_stop_condition_matches_the_mse_branch():
    """stop_condition is the criterion nmf_multupdate_mse evaluates: the same iteration count on the same problem."""
    rng = np.random.default_rng(5)
    X = rng.random((20, 15))
    W0, H0 = rng.random((20, 3)), rng.random((3, 15))
    inf = {}
    o.nmf_multupdate_mse(X, 3, Winit=W0, Hinit=H0, maxiter=2000, tol=1e-3, info=inf)
    W, H, n = W0.copy(), H0.copy(), 0
    while True:
        n += 1
        preW, preH = W.copy(), H.copy()
        H *= (W.T @ X) / ((W.T @ W) @ H + multupdate_div_delta(np.float64))
        W *= (X @ H.T) / (W @ (H @ H.T) + multupdate_div_delta(np.float64))
        if stop_condition(W, preW, H, preH, 1e-3) or n >= 2000:
            break
    assert n == inf["iters"] and inf["converged"]


def test_delta_zero_matches_nmf_multiplicative_until_the_first_clamp():
    """With delta = 0 on strictly positive X the update is NMFmultiplicative's (NMFkMultiplicative.jl:67,70); the two differ
    from iteration 10 on, where NMFmultiplicative clamps the factors (:99-100)."""
    rng = np.random.default_rng(7)
    n, m, k = 30, 20, 4
    X = rng.random((n, m)) + 0.1
    W0 = rng.random((n, k))
    H0 = rng.random((k, m))
    ref, div = [], []
    o.nmf_multiplicative(X.copy(), k, Winit=W0.copy(), Hinit=H0.copy(), maxiter=12, tolOF=-1.0,
                         trace=lambda it, W, H, obj: ref.append((W.copy(), H.copy())))
    nmf_multupdate_div(X, k, Winit=W0, Hinit=H0, maxiter=12, tol=0.0, delta=0.0,
                       trace=lambda it, W, H: div.append((W.copy(), H.copy())))
    assert len(ref) == len(div) == 12
    for t in range(9):
        assert np.array_equal(ref[t][0], div[t][0]) and np.array_equal(ref[t][1], div[t][1]), t


def test_default_delta_is_sqrt_eps_of_the_data_type():
    assert multupdate_div_delta(np.float64) == 2.0 ** -26
    assert multupdate_div_delta(np.float32) == float(np.float32(np.sqrt(np.float32(2.0 ** -23))))


def test_stop_rule_hand_checked():
    """X = w h with a rank-one factorisation that is already a fixed point of the delta = 0 update: the factors do not move,
    so stop_condition holds after the first iteration for any tol >= 0.  Scaling H by 2 breaks the fixed point: the first
    update moves every row of H by |2 - 1| / (2 + 1) = 1/3 relative (W by 0), so tol = 0.34 stops after one iteration and
    tol = 0.33 does not."""
    w = np.array([[1.0], [2.0], [3.0]])
    h = np.array([[1.0, 1.0, 2.0, 4.0]])
    X = w @ h
    inf = {}
    W, H, gkl = nmf_multupdate_div(X, 1, Winit=w / w.sum(), Hinit=h * w.sum(), maxiter=50, tol=0.0, delta=0.0, info=inf)
    assert inf == {"iters": 1, "converged": True, "stop_reason": "tol"}
    assert abs(gkl) < 1e-12
    for tol, iters in ((0.34, 1), (0.33, 2)):
        inf = {}
        nmf_multupdate_div(X, 1, Winit=w / w.sum(), Hinit=2 * h * w.sum(), maxiter=50, tol=tol, delta=0.0, info=inf)
        assert inf["iters"] == iters and inf["converged"], (tol, inf)


def test_zeros_of_x_stay_zeros_and_maxiter_stops():
    """No lambda substitution: an all-zero column of X gives a zero column of H after the first update."""
    rng = np.random.default_rng(3)
    X = rng.random((12, 9))
    X[:, 4] = 0.0
    inf = {}
    W, H, _ = nmf_multupdate_div(X, 3, Winit=rng.random((12, 3)), Hinit=rng.random((3, 9)), maxiter=5, tol=0.0, info=inf)
    assert inf == {"iters": 5, "converged": False, "stop_reason": "maxiter"}
    assert np.all(H[:, 4] == 0.0) and np.all(H[:, [0, 1, 2, 3, 5, 6, 7, 8]] > 0)
    W2, H2, obj = execute_singlerun_nmf_multmse(X, 3, Winit=W, Hinit=H, maxiter=1)
    assert np.allclose(H2[[0, 1, 2]].sum(axis=1), 1.0)
