"""Host-side mirror of the reference's Julia interface for the hot path.

Every public function cites the reference method it stands for (paths relative to
/root/reference/src).  Arrays are NumPy, column-major (Fortran order) like Julia's; nothing
numeric happens here - all of it is a call into the C ABI (libnmfk_b200.so)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import F32, F64, NMFkError, Params, XInfo, check

_DT = {np.dtype(np.float32): F32, np.dtype(np.float64): F64}
_NP = {F32: np.float32, F64: np.float64}


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f(a, dtype) -> np.ndarray:
    return np.asfortranarray(a, dtype=dtype)


def default_params(**kw) -> Params:
    """Keyword defaults as reached from NMFk.execute(...; method=:simple)
    (NMFkExecute.jl:729 -> NMFkMultiplicative.jl:24)."""
    p = Params()
    _lib.load().nmfk_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError("unknown solver parameter %r" % k)
        setattr(p, k, v)
    return p


class Context:
    """One CUDA device + one data matrix X (nmfk_ctx)."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        check(self._lib.nmfk_ctx_create(device, C.byref(h)))
        self._h = h
        self.dtype = None
        self.n = self.m = 0

    def close(self):
        if getattr(self, "_h", None):
            self._lib.nmfk_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_X(self, X: np.ndarray, lam: float = 1e-32, normalizevector=None):
        """NMFpreprocessing! (NMFkMultiplicative.jl:3-22).  The caller's X is never modified.
        normalizevector (length n, :27-31): the solver works on X ./ normalizevector, W is scaled back and the objective is
        taken against X itself when a restart finishes (:119-125)."""
        X = np.asarray(X)
        if X.ndim != 2:
            raise ValueError("X must be a matrix (N>2 arrays are delegated to tensorfactorization in the reference)")
        if X.dtype not in _DT:
            X = X.astype(np.float64)
        Xf = np.asfortranarray(X)
        self.dtype = _DT[Xf.dtype]
        self.np_dtype = Xf.dtype.type
        self.n, self.m = Xf.shape
        nv = None
        if normalizevector is not None and len(normalizevector) != 0:
            nv = np.ascontiguousarray(np.asarray(normalizevector, dtype=self.np_dtype).reshape(-1))
            if nv.shape[0] != self.n:  # :30
                raise NMFkError(-4, "Length of normalizing vector does not match: %d vs %d" % (nv.shape[0], self.n))
        check(self._lib.nmfk_set_X(self._h, _ptr(Xf), self.n, self.m, self.dtype, lam, _ptr(nv), 0), self._h)
        return self.xinfo()

    def set_weight(self, weight):
        """The `weight` keyword when it is an array (NMFkExecute.jl:484): a vector of length n weights the rows, a 1 x m
        matrix the columns, an n x m matrix the entries of (X - W*H) in the objective (NMFkMultiplicative.jl:74,125).
        None or a scalar clears it (scalars travel in the solver parameters)."""
        if weight is None or np.isscalar(weight):
            check(self._lib.nmfk_set_weight(self._h, None, 0, 0), self._h)
            return
        w = np.asarray(weight, dtype=self.np_dtype)
        if w.ndim == 1:
            w = w.reshape(-1, 1)  # a Julia Vector broadcasts as a column
        wf = np.asfortranarray(w)
        check(self._lib.nmfk_set_weight(self._h, _ptr(wf), wf.shape[0], wf.shape[1]), self._h)

    def comm_init(self, nranks: int, rank: int, unique_id: Optional[bytes], row0: int, n_global: int):
        """Row-sharded X (BASELINE C5; NMFmultiplicative(::DArray), NMFkMultiplicative.jl:129-197): this
        context holds rows [row0, row0 + n_local) of an n_global x m matrix, H is replicated, the tiled
        engine all-reduces the k x m numerators every iteration.  unique_id: 128 bytes from
        `comm_unique_id()` on one rank (None with nranks == 1: same code path, no NCCL)."""
        buf = None
        if unique_id is not None:
            assert len(unique_id) == 128
            buf = C.create_string_buffer(bytes(unique_id), 128)
        check(self._lib.nmfk_ctx_comm_init(self._h, int(nranks), int(rank), buf, int(row0), int(n_global)), self._h)

    def xinfo(self) -> XInfo:
        xi = XInfo()
        check(self._lib.nmfk_get_xinfo(self._h, C.byref(xi)), self._h)
        return xi

    def batch(self, k: int, R: int) -> "Batch":
        return Batch(self, k, R)

    def import_solutions(self, H: np.ndarray, obj_norm, W: Optional[np.ndarray] = None, iters=None) -> "Batch":
        """A batch made of finished solutions (nmfk_batch_create_hstack / nmfk_batch_create + nmfk_batch_import): H (R, k, m),
        optional W (R, n, k), objective values (NMFkExecute.jl:792) - the input of `Batch.cluster` without a solve, e.g.
        solutions gathered from other ranks or loaded from a result file."""
        H = np.asarray(H, dtype=self.np_dtype)
        R, k, m = H.shape
        assert m == self.m
        b = Batch.__new__(Batch)
        b.ctx, b.k, b.R = self, int(k), int(R)
        h = C.c_void_p()
        if W is None:
            check(self._lib.nmfk_batch_create_hstack(self._h, b.k, b.R, C.byref(h)), self._h)
        else:
            check(self._lib.nmfk_batch_create(self._h, b.k, b.R, C.byref(h)), self._h)
        b._h = h
        Hs = np.ascontiguousarray(np.transpose(H, (0, 2, 1)))
        Ws = None if W is None else np.ascontiguousarray(np.transpose(np.asarray(W, dtype=self.np_dtype), (0, 2, 1)))
        ob = np.ascontiguousarray(obj_norm, dtype=np.float64)
        it = np.zeros(R, dtype=np.int32) if iters is None else np.ascontiguousarray(iters, dtype=np.int32)
        check(self._lib.nmfk_batch_import(h, _ptr(Ws), _ptr(Hs), ob.ctypes.data_as(_lib._pdbl), it.ctypes.data_as(_lib._pi32), 0),
              self._h)
        return b

    def solve(self, batches: Sequence["Batch"], params: Optional[Params] = None):
        """The restart loop of execute_run for all batches at once (NMFkExecute.jl:510-544)."""
        p = params or default_params()
        arr = (C.c_void_p * len(batches))(*[b._h for b in batches])
        check(self._lib.nmfk_solve(self._h, arr, len(batches), C.byref(p)), self._h)

    @property
    def launches(self) -> int:
        return int(self._lib.nmfk_launch_count(self._h))

    @property
    def last_solve_ms(self) -> float:
        return float(self._lib.nmfk_last_solve_ms(self._h))

    def profile(self, on: bool = True):
        """Time the pass-kernel launches of the tiled engine with CUDA events (nmfk_profile_enable; resets the counters)."""
        check(self._lib.nmfk_profile_enable(self._h, int(on)), self._h)

    def profile_get(self):
        """-> (summed device ms of the pass-kernel launches, number of launches) since `profile()`."""
        ms, cnt = C.c_double(), C.c_int64()
        check(self._lib.nmfk_profile_get(self._h, C.byref(ms), C.byref(cnt)), self._h)
        return ms.value, cnt.value

    def gemm_nt(self, A: np.ndarray, B: np.ndarray, reps: int = 1):
        """C = A @ B.T with the stacked-restart GEMM of Variant FRO (nmfk_gemm_nt): A (M, K), B (N, K) C-contiguous, Float32
        (tcgen05 3xTF32) or Float64 (DMMA).  -> (C (M, N), average device ms per launch)."""
        dt = np.float32 if A.dtype == np.float32 else np.float64
        A = np.ascontiguousarray(A, dtype=dt)
        B = np.ascontiguousarray(B, dtype=dt)
        M, K = A.shape
        N = B.shape[0]
        assert B.shape[1] == K
        Cm = np.empty((M, N), dtype=dt)
        ms = C.c_double()
        check(self._lib.nmfk_gemm_nt(self._h, _DT[np.dtype(dt)], _ptr(A), _ptr(B), M, N, K, _ptr(Cm), int(reps), C.byref(ms)), self._h)
        return Cm, ms.value

    def fit(self, W: np.ndarray, H: np.ndarray) -> float:
        """normnan(X - W*H) with NaN residuals zeroed (NMFkExecute.jl:664-668, :212-222) for host factors W (n,k), H (k,m)."""
        Wf, Hf = _f(W, self.np_dtype), _f(H, self.np_dtype)
        k = Wf.shape[1]
        assert Wf.shape == (self.n, k) and Hf.shape == (k, self.m)
        phi = C.c_double()
        check(self._lib.nmfk_fit(self._h, k, _ptr(Wf), _ptr(Hf), C.byref(phi)), self._h)
        return phi.value

    def measure_peak(self, which: int) -> float:
        v = C.c_double()
        check(self._lib.nmfk_measure_peak(self._h, which, C.byref(v)), self._h)
        return v.value


def comm_unique_id() -> bytes:
    """128-byte NCCL unique id (ncclGetUniqueId); send it to the other ranks by any side channel."""
    buf = C.create_string_buffer(128)
    check(_lib.load().nmfk_comm_unique_id(buf))
    return buf.raw


class Batch:
    """R restarts at one k with device-resident factor stacks (nmfk_batch)."""

    def __init__(self, ctx: Context, k: int, R: int):
        self.ctx, self.k, self.R = ctx, int(k), int(R)
        h = C.c_void_p()
        check(ctx._lib.nmfk_batch_create(ctx._h, self.k, self.R, C.byref(h)), ctx._h)
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            self.ctx._lib.nmfk_batch_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_init(self, Winit=None, Hinit=None, seed0: int = 0):
        """Winit: (R, n, k) or list of n x k; Hinit: (R, k, m).  Sizes are asserted like NMFkMultiplicative.jl:40,50.
        Either may be None: that factor is then drawn on the device from restart r's Philox stream (key seed0 + r + 1),
        the first numbers of the stream when it is the only one drawn (:37-55)."""
        c = self.ctx
        Wb = Hb = None
        if Winit is not None:
            W = np.stack([_f(w, c.np_dtype) for w in Winit]) if not isinstance(Winit, np.ndarray) else Winit
            assert W.shape == (self.R, c.n, self.k), "size(Winit) == (n, k)"
            Wb = np.ascontiguousarray(np.transpose(W, (0, 2, 1)), dtype=c.np_dtype)  # restart-major stack of column-major matrices
        if Hinit is not None:
            H = np.stack([_f(h, c.np_dtype) for h in Hinit]) if not isinstance(Hinit, np.ndarray) else Hinit
            assert H.shape == (self.R, self.k, c.m), "size(Hinit) == (k, m)"
            Hb = np.ascontiguousarray(np.transpose(H, (0, 2, 1)), dtype=c.np_dtype)
        check(c._lib.nmfk_batch_set_init_partial(self._h, _ptr(Wb), _ptr(Hb), int(seed0)), c._h)

    def init_random(self, seed0: int):
        check(self.ctx._lib.nmfk_batch_init_random(self._h, int(seed0)), self.ctx._h)

    def get(self, factors: bool = True):
        """-> dict(W (R,n,k), H (R,k,m), obj_ssq, obj_norm, iters, stop_reason)."""
        c = self.ctx
        R, k = self.R, self.k
        out = {}
        Wb = np.empty((R, k, c.n), dtype=c.np_dtype) if factors else None
        Hb = np.empty((R, c.m, k), dtype=c.np_dtype) if factors else None
        ssq = np.empty(R)
        nrm = np.empty(R)
        it = np.empty(R, dtype=np.int32)
        sr = np.empty(R, dtype=np.int32)
        check(c._lib.nmfk_batch_get(self._h, _ptr(Wb), _ptr(Hb), ssq.ctypes.data_as(_lib._pdbl),
                                    nrm.ctypes.data_as(_lib._pdbl), it.ctypes.data_as(_lib._pi32),
                                    sr.ctypes.data_as(_lib._pi32)), c._h)
        if factors:
            out["W"] = np.transpose(Wb, (0, 2, 1))  # views: (R, n, k) with column-major matrices
            out["H"] = np.transpose(Hb, (0, 2, 1))
        out.update(obj_ssq=ssq, obj_norm=nrm, iters=it, stop_reason=sr)
        return out

    def objective(self, weight: float = 1.0) -> np.ndarray:
        o = np.empty(self.R)
        check(self.ctx._lib.nmfk_batch_objective(self._h, weight, o.ctypes.data_as(_lib._pdbl)), self.ctx._h)
        return o

    def select(self, acceptratio: float = 1, acceptfactor: float = np.inf, nanaction: str = "zeroed"):
        """Solution filtering of execute_run (NMFkExecute.jl:551-597): -> sorted restart indices that reach
        clustersolutions / finalize.  Stored in the batch; `cluster` / `cluster_means` then work on them."""
        if nanaction not in ("zeroed", "removed"):
            raise NMFkError(-1, "nanaction must be :zeroed or :removed")
        order = np.empty(self.R, dtype=np.int32)
        nk = C.c_int32()
        check(self.ctx._lib.nmfk_batch_select(self._h, float(acceptratio), float(acceptfactor), int(nanaction == "removed"),
                                              order.ctypes.data_as(_lib._pi32), C.byref(nk)), self.ctx._h)
        self.nkept = nk.value
        return order[:nk.value].copy()

    def cluster(self, clusterWmatrix: bool = False):
        """sortperm + clustersolutions + finalize silhouettes (NMFkExecute.jl:545-638,
        NMFkCluster.jl:425-517, NMFkFinalize.jl:36-79).
        -> dict(order (R,), labels (k,R) 1-based, sil (k,R), clustersil (k,), robustness, centroids)."""
        c = self.ctx
        R, k = self.R, self.k
        order = np.empty(R, dtype=np.int32)
        labels = np.empty((R, k), dtype=np.int32)
        sil = np.empty((R, k))
        csil = np.empty(k)
        rob = C.c_double()
        ln = c.n if clusterWmatrix else c.m
        cent = np.zeros((ln + 1, k), dtype=c.np_dtype)
        cols = C.c_int32()
        check(c._lib.nmfk_batch_cluster(self._h, int(clusterWmatrix), order.ctypes.data_as(_lib._pi32),
                                        labels.ctypes.data_as(_lib._pi32), sil.ctypes.data_as(_lib._pdbl),
                                        csil.ctypes.data_as(_lib._pdbl), C.byref(rob), _ptr(cent), C.byref(cols)), c._h)
        nk = getattr(self, "nkept", None) or R  # after select(): only the kept solutions were clustered
        return dict(order=order[:nk], labels=labels[:nk].T, sil=sil[:nk].T, clustersil=csil, robustness=rob.value,
                    centroids=cent[:cols.value].T if cols.value else None)


    def cluster_means(self, order: np.ndarray, labels: np.ndarray):
        """Wmean, Hmean, Wvar, Hvar of finalize (NMFkFinalize.jl:68-74) from the outputs of `cluster()`:
        -> dict(W (n,k), H (k,m), Wvar (n,k), Hvar (k,m))."""
        c = self.ctx
        k = self.k
        order = np.ascontiguousarray(order, dtype=np.int32)
        lab = np.ascontiguousarray(np.asarray(labels, dtype=np.int32).T)  # (R, k): column-major k x R
        Wm, Wv = np.empty((k, c.n), dtype=c.np_dtype), np.empty((k, c.n), dtype=c.np_dtype)
        Hm, Hv = np.empty((c.m, k), dtype=c.np_dtype), np.empty((c.m, k), dtype=c.np_dtype)
        check(c._lib.nmfk_batch_cluster_means(self._h, order.ctypes.data_as(_lib._pi32), lab.ctypes.data_as(_lib._pi32),
                                              _ptr(Wm), _ptr(Hm), _ptr(Wv), _ptr(Hv)), c._h)
        return dict(W=Wm.T, H=Hm.T, Wvar=Wv.T, Hvar=Hv.T)


# ------------------------------------------------------------------------------------------
# reference-shaped functions
# ------------------------------------------------------------------------------------------
_PARAM_NAMES = ("tol", "tolOF", "maxiter", "maxbaditers", "maxreattempts", "stopconv", "Wfixed", "Hfixed", "engine", "iter_limit",
                "normalize", "stop_rule", "variant")


def _params_from_kw(kw: dict, ctx: Optional[Context] = None, **defaults) -> Params:
    """Map the reference's keyword names onto nmfk_params; unknown keywords are tolerated like the `kw...` sink of
    NMFkMultiplicative.jl:24.  `weight`: a scalar travels in the parameters, an array (vector of length n, 1 x m, n x m;
    NMFkExecute.jl:484) is installed on the context."""
    vals = dict(defaults)
    method = str(kw.pop("method", "simple")).lstrip(":")
    algorithm = str(kw.pop("algorithm", "multdiv")).lstrip(":")
    if method == "nmf":  # NMFkExecute.jl:763-775: NMF.jl solvers, names swapped in the reference (:765-768):
        # :multdiv is MultUpdate(obj=:mse) = Variant FRO, :multmse is MultUpdate(obj=:div) = Variant KL_DIV
        if algorithm == "multdiv":
            vals["variant"] = 1
        elif algorithm == "multmse":
            vals["variant"] = 3
        else:
            raise NMFkError(-6, "method=:nmf: only algorithm=:multdiv and :multmse (NMF.MultUpdate) are on the B200 path")
    elif method == "sparsity":  # NMFkExecute.jl:757-758: NMFsparsity(Xn, nk; maxiter, tol, kw...)
        if ctx is None:
            raise NMFkError(-1, "method=:sparsity needs a context")
        beta = kw.pop("beta_divergence", -1)
        cf = str(kw.pop("cost_function", "ed")).lstrip(":")
        if beta == -1:  # NMFkSparsity.jl:5-22
            beta = {"kl": 1, "ed": 2, "is": 0}.get(cf, 2)
        check(ctx._lib.nmfk_set_sparsity_options(ctx._h, float(beta), float(kw.pop("sparsity", 1)), float(kw.pop("lam_sparsity", 1e-9))),
              ctx._h)
        vals["variant"] = 2
    elif method != "simple":
        raise NMFkError(-6, "method=:%s is not on the B200 path (:simple, :sparsity and :nmf with algorithm=:multdiv or :multmse "
                            "are)" % method)
    for k in list(kw):
        if k in _PARAM_NAMES:
            vals[k] = kw.pop(k)
    weight = kw.pop("weight", vals.pop("weight", 1))
    if np.isscalar(weight):
        vals["weight"] = float(weight)
        if ctx is not None:
            ctx.set_weight(None)
    else:
        if ctx is None:
            raise NMFkError(-1, "array weights need a context")
        vals["weight"] = 1.0
        ctx.set_weight(weight)
    for b in ("Wfixed", "Hfixed"):
        if b in vals:
            vals[b] = int(bool(vals[b]))
    return default_params(**vals)


def _seed0(seed) -> int:
    """restart i (1-based) draws from Philox(key=seed+i): `seed=kwseed+i` of NMFkExecute.jl:536; no seed = the global RNG."""
    return int(seed) if seed is not None and seed >= 0 else int(np.random.randint(0, 2 ** 31))


def _stack(a, R, shape, dt, what):
    """One n x k (k x m) matrix for all restarts, like the reference's Winit / Hinit keywords, or an explicit (R, ., .) stack."""
    if a is None or np.size(a) == 0:  # sizeof(Winit) == 0 (NMFkMultiplicative.jl:37,47)
        return None
    a = np.asarray(a, dtype=dt)
    if a.ndim == 2:
        assert a.shape == shape, "size(%s) == %s" % (what, shape)  # :40,50
        a = np.broadcast_to(a, (R,) + shape)
    assert a.shape == (R,) + shape, "size(%s) == %s" % (what, shape)
    return a


def NMFmultiplicative(X, k: int, *, Winit=None, Hinit=None, seed: int = -1, lam: float = 1e-32, normalizevector=None,
                      ctx: Context = None, **kw):
    """`NMFk.NMFmultiplicative(X, k; ...)` NMFkMultiplicative.jl:24-127 -> (W, H, objvalue) with objvalue the sum of squares
    of :125.  maxiter defaults to 1000000 as in the direct call.  Winit and Hinit are independent (:37-55); weight may be a
    scalar, a vector of length n, a 1 x m or an n x m matrix (:74,125); normalizevector divides the rows of X for the solve
    (:27-31, :119-122).  (The reference substitutes lambda for zeros BEFORE dividing, so its substituted entries are
    lambda / normalizevector[i]; NaN entries here start from lambda: a 1e-32-scale difference.)"""
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X, lam, normalizevector)
        p = _params_from_kw(kw, ctx, maxiter=kw.pop("maxiter", 1000000), normalize=0)
        b = ctx.batch(k, 1)
        try:
            b.set_init(_stack(Winit, 1, (ctx.n, k), ctx.np_dtype, "Winit"), _stack(Hinit, 1, (k, ctx.m), ctx.np_dtype, "Hinit"),
                       _seed0(seed) - 1)
            ctx.solve([b], p)
            r = b.get()
        finally:
            b.close()
        return np.asfortranarray(r["W"][0]), np.asfortranarray(r["H"][0]), float(r["obj_ssq"][0])
    finally:
        if own:
            ctx.close()


def NMFsparsity(X, k: int, *, Winit=None, Hinit=None, seed: int = -1, maxiter: int = 100000, tol: float = 1e-19, lam: float = 1e-9,
                ctx: Context = None, **kw):
    """`NMFk.NMFsparsity(X, k; cost_function=:ed, beta_divergence=-1, sparsity=1, maxiter=100000, tol=1e-19, lambda=1e-9, Winit, Hinit)`
    NMFkSparsity.jl:1-113 -> (W, H, objvalue = sum((X - W*H).^2)); `lam` is the reference's `lambda` keyword."""
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X)
        p = _params_from_kw(dict(kw, method="sparsity", lam_sparsity=lam), ctx, maxiter=maxiter, tol=tol, normalize=0)
        b = ctx.batch(k, 1)
        try:
            b.set_init(_stack(Winit, 1, (ctx.n, k), ctx.np_dtype, "Winit"), _stack(Hinit, 1, (k, ctx.m), ctx.np_dtype, "Hinit"),
                       _seed0(seed) - 1)
            ctx.solve([b], p)
            r = b.get()
        finally:
            b.close()
        return np.asfortranarray(r["W"][0]), np.asfortranarray(r["H"][0]), float(r["obj_ssq"][0])
    finally:
        if own:
            ctx.close()


def NMFmultiplicative_darray(X, k: int, *, stopconv: int = 10000, **kw):
    """`NMFk.NMFmultiplicative(X::DArray, k; ...)` NMFkMultiplicative.jl:129-197: the distributed method's own stop rule (no
    tolOF / baditers / reattempts, no weight, stopconv=10000).  On one GPU this is a flag of the same engines; with the rows
    of X spread over several GPUs use nmfk_b200.dist.solve_rowsharded(..., params=default_params(stop_rule=1))."""
    kw.pop("weight", None)
    return NMFmultiplicative(X, k, stop_rule=1, stopconv=stopconv, **kw)


def execute_singlerun(X, nk: int, *, Winit=None, Hinit=None, seed: int = -1, clusterWmatrix: bool = False,
                      normalizevector=None, ctx: Context = None, **kw):
    """`execute_singlerun_compute(X, nk; method=:simple, ...)` NMFkExecute.jl:729-807 -> (W, H, objvalue): objvalue =
    normnan(X - W*H), rows of H sum to one (columns of W with clusterWmatrix=true, :796-799)."""
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X, kw.pop("lam", 1e-32), normalizevector)
        modify = kw.pop("modifymatrices", True)
        p = _params_from_kw(kw, ctx, normalize=(2 if clusterWmatrix else 1) if modify else 0)
        b = ctx.batch(nk, 1)
        try:
            b.set_init(_stack(Winit, 1, (ctx.n, nk), ctx.np_dtype, "Winit"), _stack(Hinit, 1, (nk, ctx.m), ctx.np_dtype, "Hinit"),
                       _seed0(seed) - 1)
            ctx.solve([b], p)
            r = b.get()
        finally:
            b.close()
        return np.asfortranarray(r["W"][0]), np.asfortranarray(r["H"][0]), ctx.np_dtype(r["obj_norm"][0])
    finally:
        if own:
            ctx.close()


def _run_inits(ctx, nk, nNMF, inits, Winit, Hinit):
    """(Winit stack, Hinit stack) from either the harness-style `inits=(W (R,n,k), H (R,k,m))` or the reference's single
    Winit / Hinit matrices shared by every restart (the kw pass-through of NMFkExecute.jl:536)."""
    if inits is not None:
        Winit, Hinit = inits
    return (_stack(Winit, nNMF, (ctx.n, nk), ctx.np_dtype, "Winit"), _stack(Hinit, nNMF, (nk, ctx.m), ctx.np_dtype, "Hinit"))


def execute_run(X, nk: int, nNMF: int, *, clusterWmatrix: bool = False, seed: Optional[int] = None, inits=None, Winit=None,
                Hinit=None, ctx: Context = None, details: Optional[dict] = None, best: bool = True, acceptratio: float = 1,
                acceptfactor: float = np.inf, nanaction: str = "zeroed", normalizevector=None, **kw):
    """`execute_run(X, nk, nNMF; ...)` NMFkExecute.jl:483-711 -> (Wa, Ha, phi, minsilhouette, aic).
    clusterWmatrix selects the stack that is clustered (:620-624) and is NOT forwarded to the restarts (:516-540).
    best=False returns the per-cluster means of `finalize` (:637, :646-650) instead of the best restart;
    acceptratio / acceptfactor / nanaction filter the solutions that reach clustersolutions (:551-597).
    `seed`: restart i draws from Philox(key=seed+i) (the `seed=kwseed+i` of :536); Winit / Hinit (one matrix for all restarts,
    independently, like the reference) or `inits=(Winit (R,n,k), Hinit (R,k,m))` inject explicit initialisations.
    details (dict) receives the fields of the "-all" result file (:650-654)."""
    import math
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X, kw.pop("lam", 1e-32), normalizevector)
        modify = not ("Wfixed" in kw or "Hfixed" in kw)  # :486-489
        p = _params_from_kw(kw, ctx, normalize=1 if modify else 0, clusterWmatrix=int(bool(clusterWmatrix)))
        n, m, dt = ctx.n, ctx.m, ctx.np_dtype
        Wi, Hi = _run_inits(ctx, nk, nNMF, inits, Winit, Hinit)
        seed0 = _seed0(seed)
        defaults = best and acceptratio >= 1 and acceptfactor == np.inf and nanaction == "zeroed" and details is None
        if defaults:  # the one-call form
            Wb = np.empty((nk, n), dtype=dt)
            Hb = np.empty((m, nk), dtype=dt)
            phi, rob, aic = C.c_double(), C.c_double(), C.c_double()
            tot = C.c_int64()
            Ws = None if Wi is None else np.ascontiguousarray(np.transpose(Wi, (0, 2, 1)))
            Hs = None if Hi is None else np.ascontiguousarray(np.transpose(Hi, (0, 2, 1)))
            check(ctx._lib.nmfk_execute_run(ctx._h, nk, nNMF, _ptr(Ws), _ptr(Hs), seed0, C.byref(p), _ptr(Wb), _ptr(Hb),
                                            C.byref(phi), C.byref(rob), C.byref(aic), C.byref(tot)), ctx._h)
            return Wb.T, Hb.T, dt(phi.value), (1 if nk == 1 else dt(rob.value)), aic.value
        # every other keyword combination: the same device calls composed here
        b = ctx.batch(nk, nNMF)
        try:
            b.set_init(Wi, Hi, seed0)
            ctx.solve([b], p)
            pre = b.get()  # Wbest / Hbest are copies taken BEFORE the NaN pass and the clustering (:549-550)
            kept = b.select(acceptratio, acceptfactor, nanaction)
            if len(kept) == 0:
                raise NMFkError(-1, "no NMF solutions remain after the acceptance filters")
            cl = b.cluster(clusterWmatrix)
            sol = b.get()
            bi = int(np.argsort(np.asarray(pre["obj_norm"], dtype=dt), kind="stable")[0])
            Wbest, Hbest = np.array(pre["W"][bi], order="F"), np.array(pre["H"][bi], order="F")
            rob = 1
            st = None
            if nk > 1:
                ci = cl["labels"][:, 0] - 1  # :631-635 reads the stored (NaN-zeroed, possibly centroid-overwritten) best
                Wbest, Hbest = np.asfortranarray(sol["W"][bi][:, ci]), np.asfortranarray(sol["H"][bi][ci, :])
                st = b.cluster_means(cl["order"], cl["labels"])
                rob = dt(cl["robustness"])
                Wa, Ha = st["W"], st["H"]
            else:  # :646-650: finalize(WBig[idxsol], HBig[idxsol]) = the first kept restart (mean over its single column / row)
                order_full = np.argsort(np.asarray(pre["obj_norm"], dtype=dt), kind="stable")
                first = int(min(np.flatnonzero(np.isin(order_full, kept))))  # idxsol is a POSITIONAL mask applied to WBig itself
                Wa, Ha = np.asfortranarray(sol["W"][first]), np.asfortranarray(sol["H"][first])
            if best:
                Wa, Ha = Wbest, Hbest
            phi = ctx.fit(Wa, Ha)
            nobs = int(np.sum(~np.isnan(np.asarray(X))))
            aic = 2 * (Wa.size + Ha.size) + nobs * math.log(phi / nobs) if phi > 0 else -math.inf
            if details is not None:
                details.update(W=sol["W"], H=sol["H"], fit=np.asarray(pre["obj_norm"], dtype=dt), order=cl["order"],
                               labels=cl["labels"] if nk > 1 else None, clustersil=cl["clustersil"] if nk > 1 else None,
                               centroids=cl["centroids"], Wmean=None if st is None else st["W"], Hmean=None if st is None else st["H"],
                               Wvar=None if st is None else st["Wvar"], Hvar=None if st is None else st["Hvar"], Wbest=Wbest,
                               Hbest=Hbest, iters=pre["iters"], total_iters=int(pre["iters"].sum()), solve_ms=ctx.last_solve_ms)
            return np.asfortranarray(Wa), np.asfortranarray(Ha), dt(phi), rob, aic
        finally:
            b.close()
    finally:
        if own:
            ctx.close()


def execute_k(X, nk: int, nNMF: int = 10, *, ordersignals: bool = True, load: bool = False, save: bool = False, loadonly: bool = False,
              resultdir: str = ".", casefilename: str = "nmfk", **kw):
    """`NMFk.execute(X, nk::Integer, nNMF; ...)` NMFkExecute.jl:236-329 -> (W[:, so], H[so, :], fitquality, robustness, aic).
    load / save / loadonly / resultdir / casefilename drive the result cache exactly like the reference (nmfk_b200.cache; the
    reference defaults load = save = true, this mirror defaults them to false so that nothing is written unasked)."""
    if np.size(X) == 0:
        raise NMFkError(-7, "Input array has a zero dimension!")  # :242-244
    if load or save or loadonly:
        from . import cache
        return cache.execute_k_cached(X, nk, nNMF, runner=execute_run, signalorder=signalorder, resultdir=resultdir,
                                      casefilename=casefilename, loadonly=loadonly, load=load, save=save, ordersignals=ordersignals, **kw)
    if "Wfixed" in kw or "Hfixed" in kw:  # :305-307
        ordersignals = False
    W, H, fit, rob, aic = execute_run(X, nk, nNMF, **kw)
    so = signalorder(W, H) if ordersignals else np.arange(W.shape[1])  # :311-318
    return np.asfortranarray(W[:, so]), np.asfortranarray(H[so, :]), fit, rob, aic


def execute(X, nkrange, nNMF: int = 10, *, cutoff: float = 0.5, seed: Optional[int] = None, inits=None, Winit=None, Hinit=None,
            clusterWmatrix: bool = False, normalizevector=None, ctx: Context = None, details: Optional[dict] = None, **kw):
    """`NMFk.execute(X, nkrange, nNMF; cutoff=0.5, method=:simple, ...)` NMFkExecute.jl:178-233 without
    the JLD cache -> (W, H, fitquality, robustness, aic, kopt).  W, H are dicts keyed by k (the
    reference's Vector indexed by k); fitquality/robustness/aic have length maximum(nkrange) with
    fitquality[1]=Inf, robustness[1]=-1 (:200-201); kopt is k, 0 or None (`nothing`).
    All k of the range are solved concurrently on the device.  `inits[k] = (Winit (R,n,k), Hinit (R,k,m))` injects per-restart
    initial factors (either entry may be None)."""
    if isinstance(nkrange, (int, np.integer)):
        return execute_k(X, int(nkrange), nNMF, seed=seed, inits=inits, Winit=Winit, Hinit=Hinit, clusterWmatrix=clusterWmatrix,
                         normalizevector=normalizevector, ctx=ctx, **kw)
    ks = [int(k) for k in nkrange]
    if (Winit is not None or Hinit is not None) and len(ks) > 1:
        raise NMFkError(-4, "Winit / Hinit fix one k: size(Winit) == (n, k) (NMFkMultiplicative.jl:40,50)")
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X, kw.pop("lam", 1e-32), normalizevector)
        modify = not ("Wfixed" in kw or "Hfixed" in kw)
        p = _params_from_kw(kw, ctx, normalize=1 if modify else 0, clusterWmatrix=int(bool(clusterWmatrix)))
        n, m, dt = ctx.n, ctx.m, ctx.np_dtype
        nks = len(ks)
        Wo = [np.empty((k, n), dtype=dt) for k in ks]
        Ho = [np.empty((m, k), dtype=dt) for k in ks]
        Wop = (C.c_void_p * nks)(*[w.ctypes.data for w in Wo])
        Hop = (C.c_void_p * nks)(*[h.ctypes.data for h in Ho])
        Wi_keep, Hi_keep = [], []
        Wip = Hip = None
        if inits is not None or Winit is not None or Hinit is not None:
            for k in ks:
                Wi, Hi = _run_inits(ctx, k, nNMF, None if inits is None else inits[k], Winit, Hinit)
                Wi_keep.append(None if Wi is None else np.ascontiguousarray(np.transpose(Wi, (0, 2, 1))))
                Hi_keep.append(None if Hi is None else np.ascontiguousarray(np.transpose(Hi, (0, 2, 1))))
            Wip = (C.c_void_p * nks)(*[None if w is None else w.ctypes.data for w in Wi_keep])
            Hip = (C.c_void_p * nks)(*[None if h is None else h.ctypes.data for h in Hi_keep])
        fit = np.empty(nks)
        rob = np.empty(nks)
        aic = np.empty(nks)
        kopt = C.c_int32()
        tot = C.c_int64()
        karr = np.asarray(ks, dtype=np.int32)
        check(ctx._lib.nmfk_execute(ctx._h, karr.ctypes.data_as(_lib._pi32), nks, nNMF, Wip, Hip, _seed0(seed), C.byref(p),
                                    cutoff, Wop, Hop, fit.ctypes.data_as(_lib._pdbl), rob.ctypes.data_as(_lib._pdbl),
                                    aic.ctypes.data_as(_lib._pdbl), C.byref(kopt), C.byref(tot)), ctx._h)
        maxk = max(ks)
        fitquality = np.zeros(maxk, dtype=dt)
        robustness = np.zeros(maxk, dtype=dt)
        aicv = np.zeros(maxk, dtype=dt)
        fitquality[0] = np.inf  # :200
        robustness[0] = -1  # :201
        W, H = {}, {}
        for i, k in enumerate(ks):
            W[k], H[k] = Wo[i].T, Ho[i].T
            fitquality[k - 1], robustness[k - 1], aicv[k - 1] = fit[i], (1 if k == 1 else rob[i]), aic[i]
        if details is not None:
            details.update(total_iters=tot.value, solve_ms=ctx.last_solve_ms, launches=ctx.launches)
        ko = kopt.value
        return W, H, fitquality, robustness, aicv, (None if ko < 0 else ko)
    finally:
        if own:
            ctx.close()


class KmeansResult:
    """The fields of Clustering.KmeansResult that robustkmeans returns (after sortclustering)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def kmeanspp_seeds(X: np.ndarray, k: int, rng: np.random.Generator) -> np.ndarray:
    """k-means++ seeding as Clustering.kmeans does it by default (`initseeds(:kmpp, X, k)`: squared Euclidean costs whatever the
    clustering distance): first seed uniform, the next ones sampled with probability proportional to the cost to the closest
    seed so far.  The reference draws from Julia's RNG; here from `rng` (0-based point indices)."""
    d, n = X.shape
    seeds = np.empty(k, dtype=np.int32)
    seeds[0] = rng.integers(n)
    cost = np.sum((X - X[:, [seeds[0]]]) ** 2, axis=0)
    for q in range(1, k):
        tot = cost.sum()
        seeds[q] = rng.choice(n, p=cost / tot) if tot > 0 else rng.integers(n)
        cost = np.minimum(cost, np.sum((X - X[:, [seeds[q]]]) ** 2, axis=0))
    return seeds


def robustkmeans(X, k, repeats: int = 1000, *, maxiter: int = 1000, tol: float = 1e-32, compute_silhouettes_flag: bool = False,
                 best_method: str = "worst_cliff", seed: Optional[int] = None, seeds=None, ctx: Context = None, details: Optional[dict] = None):
    """`NMFk.robustkmeans(X, k, repeats; maxiter, tol, distance=CosineDist(), compute_silhouettes_flag)` NMFkCluster.jl:172-246 and,
    with a range of k, :138-170 (best_method :worst_cliff / :worst_cluster_cliff).  X is d x N with the points in the COLUMNS.
    All repeats run concurrently on the device (nmfk_robustkmeans); the k-means++ seeds come from NumPy's Philox(seed) here
    (Julia's RNG in the reference) or explicitly as `seeds` (repeats, k).  -> KmeansResult, or (KmeansResult, silhouettes)
    with compute_silhouettes_flag; None when the smallest k is not below the number of points (:139-142)."""
    own = ctx is None
    ctx = ctx or Context()
    try:
        X = np.asfortranarray(X, dtype=np.float64)
        d, N = X.shape
        if not isinstance(k, (int, np.integer)):
            krange = [int(v) for v in k]
            if krange[0] >= N:
                return None  # :139-142
            res, sil, worst, csil = {}, {}, [], []
            for q, kk in enumerate(krange):
                if kk >= N:
                    continue
                r, sl = robustkmeans(X, kk, repeats, maxiter=maxiter, tol=tol, compute_silhouettes_flag=True, seed=None if seed is None else seed + q,
                                     ctx=ctx)
                res[q], sil[q] = r, sl
                worst.append(float(np.min(sl)))
                csil.append(min(float(np.mean(sl[r.assignments == j])) for j in np.unique(r.assignments)))
            seq = worst if best_method == "worst_cliff" else csil
            if best_method not in ("worst_cliff", "worst_cluster_cliff"):
                raise NMFkError(-1, "Unknown method: best_method must be :worst_cliff or :worst_cluster_cliff")
            drops = [seq[i] - seq[i + 1] for i in range(len(seq) - 1)]
            ki = int(np.argmax(drops)) + 1  # last(findmax(...)) + 1 (:160-163)
            return res[ki]
        k = int(k)
        if seeds is None:
            rng = np.random.Generator(np.random.Philox(key=0 if seed is None else int(seed))) if seed is not None else np.random.default_rng()
            seeds = np.stack([kmeanspp_seeds(X, k, rng) for _ in range(repeats)])
        seeds = np.ascontiguousarray(seeds, dtype=np.int32)
        assert seeds.shape == (repeats, k)
        assign = np.empty(N, dtype=np.int32)
        centers = np.empty((k, d))
        costs = np.empty(N)
        counts = np.empty(k, dtype=np.int32)
        sil = np.zeros(N)
        tc = C.c_double()
        it, conv, best, nempty = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        check(ctx._lib.nmfk_robustkmeans(ctx._h, X.ctypes.data_as(_lib._pdbl), d, N, k, repeats, seeds.ctypes.data_as(_lib._pi32), maxiter,
                                         float(tol), int(compute_silhouettes_flag), assign.ctypes.data_as(_lib._pi32),
                                         centers.ctypes.data_as(_lib._pdbl), costs.ctypes.data_as(_lib._pdbl),
                                         counts.ctypes.data_as(_lib._pi32), C.byref(tc), C.byref(it), C.byref(conv),
                                         sil.ctypes.data_as(_lib._pdbl), C.byref(best), C.byref(nempty)), ctx._h)
        nc = len(np.unique(assign))
        out = KmeansResult(centers=centers.T[:, :nc], assignments=assign, costs=costs, counts=counts[:nc], totalcost=tc.value,
                           iterations=it.value, converged=bool(conv.value))
        if details is not None:
            details.update(best_repeat=best.value, empty_cluster_repeats=nempty.value)
        return (out, sil) if compute_silhouettes_flag else out
    finally:
        if own:
            ctx.close()


def getk(nkrange, robustness, cutoff: float = 0.5, strict: bool = True):
    """`getk` NMFkPostprocess.jl:7-41 -> k, 0, or None."""
    ks = np.asarray(list(nkrange), dtype=np.int32)
    rb = np.asarray(robustness, dtype=np.float64)
    if len(ks) != len(rb):
        rb = rb[ks - 1]  # :8-10
    rb = np.ascontiguousarray(rb)
    r = _lib.load().nmfk_getk(ks.ctypes.data_as(_lib._pi32), rb.ctypes.data_as(_lib._pdbl), len(ks), cutoff, int(strict))
    return None if r < 0 else int(r)


def signalorder(W, H) -> np.ndarray:
    """`signalorder` NMFkPostprocess.jl:148-158 -> 0-based order (descending contribution)."""
    W = np.asarray(W)
    dt = np.float32 if W.dtype == np.float32 else np.float64
    Wf, Hf = _f(W, dt), _f(H, dt)
    n, k = Wf.shape
    assert Hf.shape[0] == k
    o = np.empty(k, dtype=np.int32)
    check(_lib.load().nmfk_signalorder(_ptr(Wf), _ptr(Hf), n, k, Hf.shape[1], _DT[np.dtype(dt)],
                                       o.ctypes.data_as(_lib._pi32)))
    return o


def trace(X, k: int, Winit, Hinit, niter: int, *, ctx: Context = None, **kw):
    """Per-iteration dump for parity tests (nmfk_trace): -> (W_t (niter,n,k), H_t (niter,k,m), obj_t)."""
    own = ctx is None
    ctx = ctx or Context()
    try:
        ctx.set_X(X, kw.pop("lam", 1e-32))
        p = _params_from_kw(kw, ctx, normalize=0, maxiter=kw.pop("maxiter", 1000000))
        n, m, dt = ctx.n, ctx.m, ctx.np_dtype
        Wi, Hi = _f(Winit, dt), _f(Hinit, dt)
        assert Wi.shape == (n, k) and Hi.shape == (k, m)
        Wt = np.empty((niter, k, n), dtype=dt)
        Ht = np.empty((niter, m, k), dtype=dt)
        ob = np.empty(niter)
        check(ctx._lib.nmfk_trace(ctx._h, k, _ptr(Wi), _ptr(Hi), C.byref(p), niter, _ptr(Wt), _ptr(Ht),
                                  ob.ctypes.data_as(_lib._pdbl)), ctx._h)
        return np.transpose(Wt, (0, 2, 1)), np.transpose(Ht, (0, 2, 1)), ob
    finally:
        if own:
            ctx.close()
