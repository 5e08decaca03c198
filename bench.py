#!/usr/bin/env python3
"""bench.py - NMF restart-iterations/sec of the B200-native NMFk hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config auto|C2|C3|C4|C5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the timed GPU path returned in its last timed step as DIR/<name>.npy (see dump_outputs): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.

Workloads (BASELINE.json `configs`, SURVEY.md 8(d); synthetic nonnegative mixtures X = W0*H0, seed 2015):
  N = 1 (default)  C3: 10000 x 10000 Float32, k = 16, nNMF = 64 - the largest single-GPU configuration.  One step = ITERS
                   iterations of all 64 restarts (fixed iteration budget, every restart active) through the tiled engine
                   (tcgen05 kind::tf32 3-term split).  X (400 MB) is larger than the 126 MB L2, so every iteration streams it.
  N > 1            C4: 100000 x 2000 Float64, k = 2:32, nNMF = 256, restarts sharded over the N GPUs (STRONG scaling: 256 / N
                   restarts of every k per GPU), fixed iteration budget, through nmfk_sweep (library-owned NCCL communicator;
                   no collective inside the iteration loop, one all-gather of H stacks + states and one W broadcast per k).
  --config C5      2,000,000 x 1000 Float32, k = 24, nNMF = 32, rows of X sharded over the N GPUs, one NCCL all-reduce of the
                   k x m x R numerators per iteration.          --config C2: 1000 x 200 Float64, execute(X, 2:10, 100), full stop rule.
value  = restart-iterations / second of the solver phase with X and the initial factors resident in HBM (device time, CUDA
         events on the library's launching stream, max over ranks).
e2e    = the same metric through the public call (C ABI: nmfk_set_X + nmfk_execute_run / nmfk_sweep) with HOST buffers: X and
         the initial factors are copied from pinned host memory, the best factors / fit / robustness / aic come back, and
         clustering + silhouettes + selection are inside the timed region.
--impl reference times the CPU restatement of the reference (oracle/nmfk_oracle.py: NumPy + OpenBLAS with the thread count SET
below, the literal operation sequence of NMFkMultiplicative.jl) on the SAME configuration; Julia itself is not installed here or
on the GPU box (SURVEY.md 0.5).  Under torchrun rank 0 alone runs it.
"""
import os

# BLAS threads of the CPU arm: set explicitly BEFORE NumPy loads OpenBLAS, identical in both arms, and not left to torchrun's
# OMP_NUM_THREADS=1 (VERDICT r1: 546 vs 996 restart-iterations/s for the same function inside one run)
BLAS_THREADS = int(os.environ.get("NMFK_BENCH_BLAS_THREADS", os.cpu_count() or 1))
os.environ["OPENBLAS_NUM_THREADS"] = str(BLAS_THREADS)
os.environ["OMP_NUM_THREADS"] = str(BLAS_THREADS)
os.environ["MKL_NUM_THREADS"] = str(BLAS_THREADS)

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402
import zlib  # noqa: E402

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "nmfk.jl_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "nmf_restart_iterations_per_sec"
UNIT = "restart-iterations/s"
SEED_X, SEED0 = 2015, 2015
# name: (n, m, k0, dtype, ks, nNMF)
CONFIGS = {
    "C2": (1000, 200, 5, np.float64, list(range(2, 11)), 100),
    "C3": (10000, 10000, 16, np.float32, [16], 64),
    "C4": (100000, 2000, 8, np.float64, list(range(2, 33)), 256),
    "C5": (2000000, 1000, 24, np.float32, [24], 32),
}
WORKLOADS = {
    "C2": "C2: synthetic mixture 1000x200 Float64 (k0=5), execute(X, 2:10, nNMF=100; method=:simple), maxiter=10000, full stop rule",
    "C3": "C3: synthetic mixture 10000x10000 Float32 (k0=16), k=16, nNMF=64, %d iterations per step with every restart active",
    "C4": "C4: synthetic mixture 100000x2000 Float64 (k0=8), k=2:32, nNMF=256 sharded over the GPUs (strong scaling), %d iterations per step",
    "C5": "C5: synthetic tall matrix 2000000x1000 Float32 (k0=24), k=24, nNMF=32, rows of X sharded over the GPUs, %d iterations per step",
}
ITERS = {"C3": 20, "C4": 3, "C5": 10}
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full` captures
TRAFFIC = {"C3": (908832000, "profiles/r02_tc2_pass_c3.txt"), "C4": (None, None), "C5": (None, None), "C2": (17534720, "profiles/r01_resident_dmma_v3_k10.txt")}


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"] or [1])
    except Exception:
        return BLAS_THREADS


def pin_blas():
    """Raise OpenBLAS to BLAS_THREADS even when the library was loaded under another setting."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=BLAS_THREADS, user_api="blas")
    except Exception:
        pass
    return blas_threads()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 << 20  # data written by --dump-outputs in all: below 64 MB with the .npy headers
BATCH_FIELDS = ("W", "H", "obj_ssq", "obj_norm", "iters", "stop_reason")  # what Batch.get returns for a solved batch


def dump_outputs(path, arrays):
    """Writes every entry of `arrays` as path/<name>.npy: Float32 arrays as Float32, everything else (Float64, counts, stop
    reasons, scalars) as Float64.  Each array gets an equal share of DUMP_BYTES; of a larger one only the entries at flat (C
    order) positions drawn from Philox(key = crc32(name)) are kept, in ascending order - the same positions in every run."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a)
        dt = np.dtype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.size * dt.itemsize > share:
            rng = np.random.Generator(np.random.Philox(key=zlib.crc32(name.encode())))
            a = a[np.unravel_index(np.sort(rng.choice(a.size, share // dt.itemsize, replace=False)), a.shape)]
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=dt))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def c5_rows(rank, world, n_global, m, k0):
    """This rank's rows of the C5 mixture: H0 from the common stream, W0 rows from a per-rank stream (16 GB of Float64 would be
    needed to build the whole matrix on every rank)."""
    r0, r1 = (n_global * rank) // world, (n_global * (rank + 1)) // world
    H0 = np.random.Generator(np.random.Philox(key=SEED_X)).random((k0, m))
    W0 = np.random.Generator(np.random.Philox(key=SEED_X + 1 + rank)).random((r1 - r0, k0))
    return np.asfortranarray((W0 @ H0).astype(np.float32)), r0, r1


# ------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle): bounded samples of the same configurations
# ------------------------------------------------------------------------------------------------------------------
_CPU_X = {}

def cpu_sample_fixed(cfg, iters, k=None, rank=0, world=1):
    """`iters` iterations of ONE restart of the configuration on the host cores (literal reference operation sequence,
    Float64 compute like the reference - SURVEY 0.4).  -> (restart-iterations, seconds)"""
    from oracle import nmfk_oracle as o
    from nmfk_b200 import synth
    n, m, k0, dt, ks, R = CONFIGS[cfg]
    k = k or ks[-1]
    scale = 4.0 if cfg == "C5" else 1.0
    if cfg not in _CPU_X:
        _CPU_X.clear()
        if cfg == "C5":
            X, _, _ = c5_rows(0, 4, n, m, k0)  # a quarter of the rows: the CPU time per iteration scales with the row count
        else:
            X = synth.mixture(n, m, k0, seed=SEED_X, dtype=dt)
        _CPU_X[cfg] = np.asfortranarray(X.astype(np.float64))
        del X
    X64 = _CPU_X[cfg]  # nmf_multiplicative restores it before returning
    nn = X64.shape[0]
    rng = np.random.Generator(np.random.Philox(key=SEED0 + 1))
    W0 = rng.random(nn * k).reshape((nn, k), order="F")
    H0 = rng.random(k * m).reshape((k, m), order="F")
    inf = {}
    t0 = time.perf_counter()
    o.nmf_multiplicative(X64, k, Winit=W0, Hinit=H0, maxiter=iters, info=inf)
    dt_s = (time.perf_counter() - t0) * scale
    return inf["iters"], dt_s


def cpu_sample_c2(iters_per_k=60):
    from oracle import nmfk_oracle as o
    from nmfk_b200 import synth
    n, m, k0, dt, ks, R = CONFIGS["C2"]
    X = synth.mixture(n, m, k0, seed=SEED_X)
    tot = 0
    t0 = time.perf_counter()
    for k in ks:
        W0, H0 = synth.philox_inits(SEED0, 1, n, k, m)
        inf = {}
        o.nmf_multiplicative(X.copy(order="F"), k, Winit=W0[0], Hinit=H0[0], maxiter=iters_per_k, info=inf)
        tot += inf["iters"]
    return tot, time.perf_counter() - t0


def cpu_step(cfg, budget_iters):
    """One bounded CPU sample of a step of `cfg` -> (restart-iterations, seconds, description)."""
    if cfg == "C2":
        tot, dt = cpu_sample_c2(60)
        return tot, dt, "60 iterations of 1 restart for each k in 2:10 (540 restart-iterations)"
    if cfg == "C4":
        tot, dt, parts = 0, 0.0, []
        it4 = budget_iters or 2
        for k in (2, 8, 16, 32):  # four k of the sweep, 1 or 2 iterations of 1 restart each
            t, d = cpu_sample_fixed("C4", it4, k=k)
            tot += t
            dt += d
            parts.append(k)
        return tot, dt, "%d iteration(s) of 1 restart at k = %s of the 2:32 sweep" % (it4, parts)
    t, d = cpu_sample_fixed(cfg, budget_iters)
    extra = " on a quarter of the rows, time x 4" if cfg == "C5" else ""
    return t, d, "%d iterations of 1 restart%s" % (budget_iters, extra)


def run_reference(args, rank, world, cfg):
    if rank != 0:
        return
    threads = pin_blas()
    # bounded samples: a long run (the driver's K) keeps the whole arm within a few minutes
    iters = {"C3": 3, "C5": 2, "C4": 2 if args.steps <= 5 else 1}.get(cfg, 0)
    for _ in range(min(args.warmup, 1)):
        cpu_step(cfg, 1 if iters else 0)
    tot, dt, what = 0, 0.0, ""
    for _ in range(args.steps):
        t, d, what = cpu_step(cfg, iters)
        tot += t
        dt += d
    val = tot / dt
    wl = WORKLOADS[cfg] % ITERS[cfg] if cfg in ITERS else WORKLOADS[cfg]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong" if cfg in ("C4", "C5") else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl, "same_config": True,
                       "note": "CPU restatement of NMFk.jl (Julia unavailable): NumPy/OpenBLAS, Float64 compute like the reference, "
                               "5 n*m*k products + 2 n*m divides per iteration, restarts serial; each step is a bounded sample "
                               "of the workload: " + what},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": what + " per step",
                             "blas_threads_set": BLAS_THREADS},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# GPU arms
# ------------------------------------------------------------------------------------------------------------------
def fixed_budget_single(ctx, nb, synth, torch, cfg, args, iters, flush, k=None, R=None, engine=2):
    """C3-style measurement on one GPU: R restarts at one k, `iters` iterations per step, every restart active."""
    n, m, k0, dt, ks, R0 = CONFIGS[cfg]
    k, R = k or ks[-1], R or R0
    f32 = dt == np.float32
    X = synth.mixture(n, m, k0, seed=SEED_X, dtype=dt)
    W0, H0 = synth.philox_inits(SEED0, R, n, k, m, dtype=dt)
    Xpin = torch.from_numpy(np.ascontiguousarray(X.T)).pin_memory()  # (m, n) C-order == n x m column-major
    Wpin = torch.from_numpy(np.ascontiguousarray(np.transpose(W0, (0, 2, 1)))).pin_memory()
    Hpin = torch.from_numpy(np.ascontiguousarray(np.transpose(H0, (0, 2, 1)))).pin_memory()
    del W0, H0
    es = 4 if f32 else 8
    h2d = (Xpin.numel() + Wpin.numel() + Hpin.numel()) * es
    d2h = (n * k + k * m) * es + 3 * 8
    # ---- device-resident arm
    ctx.set_X(X)
    params = nb.default_params(maxiter=iters, engine=engine)

    def device_step(profile, factors=False):
        b = ctx.batch(k, R)
        b.init_random(SEED0)  # the same Philox streams as the pinned host factors, generated in HBM
        if flush is not None:
            flush.fill_(1)
        torch.cuda.synchronize()
        l0 = ctx.launches
        if profile:
            ctx.profile(True)
        ctx.solve([b], params)
        ms = ctx.last_solve_ms
        pm, pl = ctx.profile_get() if profile else (0.0, 0)
        ctx.profile(False)
        out = b.get(factors=factors)
        tot = int(out["iters"].sum())
        nl = ctx.launches - l0
        b.close()
        return ms, tot, nl, pm, pl, out

    # the clock sampler starts BEFORE the warm-up steps: nvidia-smi's start-up (NVML initialisation takes driver locks) stalled
    # the launches of the first timed step in one of two runs (301 ms instead of 224 ms, profiles/r02_bench_n1_second_outlier.json);
    # the warm-up steps also create the profile events
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    for _ in range(args.warmup):
        device_step(True)
    sampler.rows.clear()  # keep the samples of the timed region only
    tot_ms = tot_it = launches = pass_l = 0
    pass_ms = 0.0
    step_ms = []
    for s in range(args.steps):
        # the factors of the last step come back only for --dump-outputs, after the solve's events have been read
        ms, tot, nl, pm, pl, out = device_step(True, factors=bool(args.dump_outputs) and s == args.steps - 1)
        step_ms.append(ms)
        tot_ms += ms
        tot_it += tot
        launches += nl
        pass_ms += pm
        pass_l += pl
    clocks = sampler.stop()

    # ---- end-to-end arm: host buffers in, best factors and scores out, through the one-call C ABI
    import ctypes as C
    Wb = np.empty((k, n), dtype=dt)
    Hb = np.empty((m, k), dtype=dt)

    def e2e_step():
        if flush is not None:
            flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.set_X(Xpin.numpy().T)  # H2D of X + preprocessing
        if os.environ.get("NMFK_TILED_TIMING"):
            print("[bench] e2e set_X %.1f ms" % ((time.perf_counter() - t0) * 1e3), file=sys.stderr)
        phi, rob, aic, tot = C.c_double(), C.c_double(), C.c_double(), C.c_int64()
        nb._lib.check(ctx._lib.nmfk_execute_run(ctx._h, k, R, C.c_void_p(Wpin.data_ptr()), C.c_void_p(Hpin.data_ptr()), SEED0,
                                                C.byref(params), Wb.ctypes.data_as(C.c_void_p), Hb.ctypes.data_as(C.c_void_p),
                                                C.byref(phi), C.byref(rob), C.byref(aic), C.byref(tot)), ctx._h)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, int(tot.value), rob.value, phi.value, aic.value

    for _ in range(min(args.warmup, 1)):
        e2e_step()
    e2e_t = e2e_it = 0
    rob = None
    for _ in range(args.steps):
        dts, t, rob, phi, aic = e2e_step()
        e2e_t += dts
        e2e_it += t
    if args.dump_outputs:  # what each arm's caller received in its last step: the batch of nmfk_solve, the best restart of nmfk_execute_run
        outputs = {name: out[name] for name in BATCH_FIELDS}
        outputs.update(e2e_W=Wb.T, e2e_H=Hb.T, e2e_fit=phi, e2e_robustness=rob, e2e_aic=aic)
        dump_outputs(args.dump_outputs, outputs)
    return dict(value=tot_it / (tot_ms * 1e-3), ms_per_step=tot_ms / args.steps, step_ms=step_ms, iters_per_step=tot_it / args.steps,
                launches=launches, pass_ms=pass_ms, pass_launches=pass_l, flops_per_pass=4.0 * n * m * k * R, clocks=clocks,
                e2e_value=e2e_it / e2e_t, e2e_ms_per_step=e2e_t / args.steps * 1e3, h2d=h2d, d2h=d2h, robustness=rob,
                n=n, m=m, k=k, R=R)


def bench_c2(ctx, nb, synth, torch, args, flush, steps, warmup, dump=None):
    """C2 on one GPU: execute(X, 2:10, 100) with the reference stop rule (the resident DMMA engine).  dump: directory for what
    the last timed step and the timed execute call returned (--dump-outputs)."""
    n, m, k0, dt, ks, R = CONFIGS["C2"]
    X = synth.mixture(n, m, k0, seed=SEED_X)
    ctx.set_X(X)
    params = nb.default_params()
    peak = max(ctx.measure_peak(1) for _ in range(2))

    def step(factors=False):
        bs = [ctx.batch(k, R) for k in ks]
        for b in bs:
            b.init_random(SEED0)
        flush.fill_(1)
        torch.cuda.synchronize()
        ctx.solve(bs, params)
        ms = ctx.last_solve_ms
        outs = {b.k: b.get(factors=factors) for b in bs}
        its = {k: int(o["iters"].sum()) for k, o in outs.items()}
        for b in bs:
            b.close()
        return ms, its, outs

    for _ in range(warmup):
        step()
    tot_ms, tot_it, flops = 0.0, 0, 0.0
    for s in range(steps):
        ms, its, outs = step(factors=bool(dump) and s == steps - 1)
        tot_ms += ms
        tot_it += sum(its.values())
        flops += sum(8.0 * n * m * k * v for k, v in its.items())
    t0 = time.perf_counter()
    W, H, fit, rob, aic, kopt = nb.execute(X, ks, R, seed=SEED0, ctx=ctx)
    e2e = time.perf_counter() - t0
    if dump:
        outputs = {"k%d_%s" % (k, name): o[name] for k, o in outs.items() for name in BATCH_FIELDS}
        for k in ks:
            outputs.update({"e2e_k%d_W" % k: W[k], "e2e_k%d_H" % k: H[k]})
        outputs.update(e2e_fit=fit, e2e_robustness=rob, e2e_aic=aic, e2e_kopt=-1 if kopt is None else kopt)
        dump_outputs(dump, outputs)
    tf = flops / (tot_ms * 1e-3) / 1e12
    return {"workload": WORKLOADS["C2"], "value": tot_it / (tot_ms * 1e-3), "unit": UNIT, "ms_per_step": tot_ms / steps,
            "restart_iterations_per_step": tot_it / steps, "kopt": kopt, "e2e_s_execute": e2e,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                         "kernel": "kl_resident_dmma_kernel<K> (one CTA per restart, DMMA m8n8k4)",
                         "peak_source": "FP64 DMMA micro-benchmark (nmfk_measure_peak 1); MEASURED_PEAKS.json has no FP64 figure"}}


def sweep_step(ctx, nbdist, torch, Xhost, ks, R_local, params, rank, world, barrier):
    barrier()
    t0 = time.perf_counter()
    out = nbdist.execute_sharded(ctx, Xhost, ks, R_local, seed0=SEED0, rank=rank, world=world, params=params)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, ctx.last_solve_ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "C2", "C3", "C4", "C5"])
    ap.add_argument("--iters", type=int, default=0, help="iterations per step of the fixed-budget configurations")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary measurements (C2, C4 on one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last timed step as DIR/<name>.npy (less than 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = args.config if args.config != "auto" else ("C3" if world == 1 else "C4")
    if args.impl == "reference":
        return run_reference(args, rank, world, cfg)

    import torch
    import nmfk_b200 as nb
    from nmfk_b200 import dist as nbdist
    from nmfk_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if use_dist:
            td.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if not use_dist:
            return list(vals)
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        td.all_reduce(t, op=td.ReduceOp.MAX)
        return t.tolist()

    def reduce_sum(vals):
        if not use_dist:
            return list(vals)
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        td.all_reduce(t, op=td.ReduceOp.SUM)
        return t.tolist()

    ctx = nb.Context(local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    mp = measured_peaks()
    iters = args.iters or ITERS.get(cfg, 0)
    line = None

    if cfg == "C3":
        if world != 1:
            raise SystemExit("bench.py: C3 is the single-GPU configuration (use --config C4 / C5 with several GPUs)")
        tf32 = max(ctx.measure_peak(13) for _ in range(3))
        ffma = max(ctx.measure_peak(2) for _ in range(2))
        r = fixed_budget_single(ctx, nb, synth, torch, "C3", args, iters, flush)
        per_launch_ms = r["pass_ms"] / max(r["pass_launches"], 1)
        achieved = r["flops_per_pass"] / (per_launch_ms * 1e-3) / 1e12
        peak = tf32 / 3.0
        traffic, traffic_src = TRAFFIC["C3"]
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOADS["C3"] % iters, "engine": "tiled; tcgen05.mma kind::tf32 3-term split, X tiles by tensor-map TMA (kl_tiled_tc2.cu)",
                       "l2": "inputs larger than L2: X is 400 MB (and its transpose another 400 MB) against 126 MB of L2; 256 MiB "
                             "are also written between steps", "restart_iterations_per_step": r["iters_per_step"],
                       "step_ms": r["step_ms"],
                       "same_config": True},
            "clocks": r["clocks"],
            "e2e": {"value": r["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "ms_per_step": r["e2e_ms_per_step"],
                    "call": "nmfk_set_X + nmfk_execute_run with pinned host X / Winit / Hinit; clustering, silhouettes and the "
                            "best-restart selection inside the timed region", "robustness": r["robustness"]},
            "gpu_launches": int(r["launches"]),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "tc2_pass_kernel<16> (one launch = one half-update of all 64 restarts)",
                         "launch_ms": per_launch_ms, "launches_timed": int(r["pass_launches"]),
                         "algorithmic_flops_per_launch": r["flops_per_pass"],
                         "algorithmic_bytes_per_launch": float(r["n"]) * r["m"] * 4,
                         "peak_source": "tcgen05.mma kind::tf32 dense throughput measured in this run by nmfk_measure_peak(13) "
                                        "(%.1f TFLOP/s) / 3 for the 3-term split; MEASURED_PEAKS.json holds bf16 %.1f TFLOP/s "
                                        "(TF32 = half of it = %.1f)" % (tf32, mp.get("bf16_tflops", float("nan")),
                                                                       mp.get("bf16_tflops", float("nan")) / 2),
                         "frac_of_fp32_ffma_peak": achieved / ffma, "fp32_ffma_peak": ffma,
                         "what_bounds": "latency, not a pipe: the 16 quotient warps (4 per scheduler) spend a unit in tensor-memory round "
                                        "trips, shared-memory loads and fixed-latency arithmetic with nothing to switch to; tensor pipe "
                                        "23 %, issue slots 64 %, no unit above 45 % (profiles/r02_tc2_pass_c3.txt, DESIGN.md 4a)",
                         "hbm_gbs_if_streaming_only": float(r["n"]) * r["m"] * 4 / (per_launch_ms * 1e-3) / 1e9,
                         "hbm_peak_gbs": mp.get("hbm_gbs")}}
        if not args.no_cpu_baseline:
            threads = pin_blas()
            t, d, what = cpu_step("C3", 6)
            line["cpu_baseline"] = {"value": t / d, "unit": UNIT, "cores": threads, "kind": "port", "blas_threads_set": BLAS_THREADS,
                                    "sample": what + " of the same configuration, oracle/nmfk_oracle.py (NumPy/OpenBLAS "
                                              "restatement of NMFkMultiplicative.jl, Float64 compute like the reference)"}
        if not args.no_also:
            line["also"] = {}
            try:
                line["also"]["C2"] = bench_c2(ctx, nb, synth, torch, args, flush, 1, 1)
            except Exception as e:
                line["also"]["C2"] = {"error": repr(e)}
            try:  # Variant FRO (method=:nmf, algorithm=:multdiv: the north star's stacked-restart GEMM) on the C3 matrix
                n, m, k0, dt, ks, R = CONFIGS["C3"]
                X3 = synth.mixture(n, m, k0, seed=SEED_X, dtype=dt)
                ctx.set_X(X3)
                pf = nb.default_params(maxiter=iters, variant=1)
                best = None
                for rep in range(3):
                    b = ctx.batch(ks[0], R)
                    b.init_random(SEED0)
                    ctx.profile(True)
                    ctx.solve([b], pf)
                    pm, pl = ctx.profile_get()
                    ctx.profile(False)
                    ms = ctx.last_solve_ms
                    tot = int(b.get(factors=False)["iters"].sum())
                    b.close()
                    if rep > 0 and (best is None or ms < best[0]):
                        best = (ms, tot, pm, pl)
                ms, tot, pm, pl = best
                gemm_tf = 2.0 * R * ks[0] * n * m * pl / (pm * 1e-3) / 1e12 if pm > 0 else float("nan")
                line["also"]["C3_variant_FRO"] = {
                    "workload": "C3 matrix, Variant FRO (NMF.jl MultUpdate(obj=:mse), NMFkExecute.jl:763-766): %d iterations of the 64 "
                                "stacked restarts" % iters, "value": tot / ms * 1e3, "unit": UNIT, "ms": ms,
                    "stacked_gemm": {"kernel": "fro_gemm_kernel (tcgen05 kind::tf32 3-term split, TMA tensor maps, cluster multicast, split-K)",
                                     "launch_ms": pm / max(pl, 1), "launches_timed": pl, "algorithmic_tflops": gemm_tf,
                                     "peak": tf32 / 3.0, "frac": gemm_tf / (tf32 / 3.0),
                                     "ncu": "profiles/r02_fro_gemm_v1.txt: sm__pipe_tensor_cycles_active 71.6 %"},
                    "note": "a different update rule than the headline (KL, method=:simple): not comparable restart-iteration for "
                            "restart-iteration in convergence, reported because the north star names this GEMM"}
                del X3
            except Exception as e:
                line["also"]["C3_variant_FRO"] = {"error": repr(e)}
            try:  # the C4 step of the multi-GPU runs on ONE GPU: the strong-scaling baseline
                n, m, k0, dt, ks, R = CONFIGS["C4"]
                X4 = synth.mixture(n, m, k0, seed=SEED_X, dtype=dt)
                p4 = nb.default_params(maxiter=ITERS["C4"], engine=2)
                ctx.profile(True)
                dt_s, solve_ms, out = sweep_step(ctx, nbdist, torch, X4, ks, R, p4, 0, 1, barrier)
                pm, pl = ctx.profile_get()
                ctx.profile(False)
                line["also"]["C4_strong_n1"] = {"workload": WORKLOADS["C4"] % ITERS["C4"], "n_gpus": 1,
                                                "value": out["total_iters"] / (solve_ms * 1e-3), "unit": UNIT, "ms_per_step": solve_ms,
                                                "e2e_value": out["total_iters"] / dt_s, "restart_iterations_per_step": out["total_iters"],
                                                "pass_ms": pm, "pass_launches": pl, "note": "one step, no warm-up"}
                del X4
            except Exception as e:
                line["also"]["C4_strong_n1"] = {"error": repr(e)}

    elif cfg == "C4":
        n, m, k0, dt, ks, R = CONFIGS["C4"]
        if R % world:
            raise SystemExit("bench.py: nNMF = 256 must be divisible by the number of GPUs")
        R_local = R // world
        X = synth.mixture(n, m, k0, seed=SEED_X, dtype=dt)
        Xpin = torch.from_numpy(np.ascontiguousarray(X.T)).pin_memory()
        del X
        params = nb.default_params(maxiter=iters, engine=2)
        dmma = max(ctx.measure_peak(1) for _ in range(2))
        sampler = ClockSampler(local_rank)
        sampler.start()  # before the warm-up: see fixed_budget_single
        for _ in range(args.warmup):
            sweep_step(ctx, nbdist, torch, Xpin.numpy().T, ks, R_local, params, rank, world, barrier)
        barrier()
        sampler.rows.clear()
        l0 = ctx.launches
        ctx.profile(True)
        wall = solve = 0.0
        its = its_local = 0
        kopt = None
        for _ in range(args.steps):
            flush.fill_(1)
            dts, sms, out = sweep_step(ctx, nbdist, torch, Xpin.numpy().T, ks, R_local, params, rank, world, barrier)
            wall += dts
            solve += sms
            its += out["total_iters"]
            its_local += out["total_iters_local"]
            kopt = out["kopt"]
        barrier()
        pm, pl = ctx.profile_get()
        ctx.profile(False)
        clocks = sampler.stop()
        launches = ctx.launches - l0
        wall_max, solve_max, pm_max = reduce_max([wall, solve, pm])
        launches_all, = reduce_sum([float(launches)])
        if rank == 0 and args.dump_outputs:  # the results of the last nmfk_sweep, the same on every rank
            outputs = {"k%d_%s" % (k, name): out[name][k] for k in ks for name in ("W", "H")}
            outputs.update(fit=out["fit"], robustness=out["robustness"], aic=out["aic"], kopt=-1 if out["kopt"] is None else out["kopt"])
            dump_outputs(args.dump_outputs, outputs)
        # the strong-scaling anchor of THIS run: rank 0 alone repeats one step with all 256 restarts of every k on its GPU (a
        # second context without the communicator) while the other ranks wait; outside the timed region
        n1 = None
        if rank == 0 and not args.no_also and args.steps <= 5:  # a long run (the driver's K) is not made 37 s longer: the one-GPU
            try:                                               # step is also in the N = 1 line (also.C4_strong_n1)
                with nb.Context(local_rank) as ctx1:
                    dt1, ms1, out1 = sweep_step(ctx1, nbdist, torch, Xpin.numpy().T, ks, R, params, 0, 1, lambda: None)
                    n1 = {"value": out1["total_iters"] / (ms1 * 1e-3), "unit": UNIT, "ms_per_step": ms1, "e2e_value": out1["total_iters"] / dt1,
                          "restart_iterations_per_step": out1["total_iters"],
                          "note": "the same step (same X, same 256 x 31 restarts, same iteration budget) on GPU 0 alone, measured in this "
                                  "run after the timed region, one step without warm-up"}
            except Exception as e:  # noqa: BLE001
                n1 = {"error": repr(e)}
        barrier()
        if rank == 0:
            flops_rank = sum(8.0 * n * m * k * R_local * iters for k in ks) * args.steps  # per GPU, both half-updates
            achieved = flops_rank / (pm_max * 1e-3) / 1e12 if pm_max > 0 else float("nan")
            es = 8
            h2d = n * m * es
            d2h = sum((n * k + k * m) * es for k in ks) + 3 * 8 * len(ks) + 12
            line = {
                "metric": METRIC, "value": its / (solve_max * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": solve_max / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOADS["C4"] % iters, "restarts_per_gpu_per_k": R_local,
                           "engine": "tiled; DMMA m8n8k4 pass (kl_tiled_dmma.cu) for k >= 4, scalar-FMA pass for k = 2, 3",
                           "sharding": "restarts (nmfk_sweep): 256 / N restarts of every k per GPU; k groups of <= 48 GB of factor stacks",
                           "l2": "inputs larger than L2: X is 1.6 GB (and its transpose); 256 MiB written between steps",
                           "restart_iterations_per_step": its / args.steps, "kopt": kopt, "same_config": True,
                           "strong_scaling_n1": n1 if n1 is not None else
                           "bench.py --gpus 1 reports this same step on one GPU under also.C4_strong_n1"},
                "clocks": clocks,
                "e2e": {"value": its / wall_max, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": wall_max / args.steps * 1e3,
                        "call": "nmfk_set_X + nmfk_sweep with pinned host X on every rank: H2D of X, device Philox initial factors, "
                                "solve, NCCL all-gather of H stacks / states, W broadcast, owner-side clustering + silhouettes, kopt"},
                "gpu_launches": int(launches_all),
                "roofline": {"bound": "tensor", "achieved": achieved, "peak": dmma, "unit": "TFLOP/s", "frac": achieved / dmma,
                             "traffic": None, "kernel": "tiled_dmma_pass_kernel<K> / tiled_pass_kernel (all k of the sweep, per GPU)",
                             "launch_ms": pm_max / max(pl, 1), "launches_timed": int(pl),
                             "peak_source": "FP64 DMMA micro-benchmark (nmfk_measure_peak 1); MEASURED_PEAKS.json has no FP64 figure",
                             "note": "achieved = 8*n*m*k flops per restart-iteration of this GPU's restarts / summed event time of "
                                     "its pass launches (slowest rank)"}}

    elif cfg == "C5":
        n, m, k0, dt, ks, R = CONFIGS["C5"]
        k = ks[0]
        Xloc, r0, r1 = c5_rows(rank, world, n, m, k0)
        uid = nbdist.exchange_unique_id(rank) if use_dist else None
        ctx.comm_init(world, rank, uid, r0, n)
        tf32 = max(ctx.measure_peak(13) for _ in range(3))
        Xpin = torch.from_numpy(np.ascontiguousarray(Xloc.T)).pin_memory()
        del Xloc
        params = nb.default_params(maxiter=iters, engine=2)

        def step(profile, factors=False):
            barrier()
            t0 = time.perf_counter()
            ctx.set_X(Xpin.numpy().T)
            b = ctx.batch(k, R)
            b.init_random(SEED0)
            if profile:
                ctx.profile(True)
            ctx.solve([b], params)
            st = b.get(factors=False)
            torch.cuda.synchronize()
            dts = time.perf_counter() - t0
            pm, pl = ctx.profile_get() if profile else (0.0, 0)
            ctx.profile(False)
            if factors:  # after the timed region: this rank's rows of W and the replicated H as well
                st = b.get()
            b.close()
            return dts, ctx.last_solve_ms, int(st["iters"].sum()), pm, pl, st

        sampler = ClockSampler(local_rank)
        sampler.start()
        for _ in range(args.warmup):
            step(True)
        barrier()
        sampler.rows.clear()
        l0 = ctx.launches
        wall = solve = pm = 0.0
        its = pl = 0
        for s in range(args.steps):
            flush.fill_(1)
            d, s_ms, t, a, b_, st = step(True, factors=rank == 0 and bool(args.dump_outputs) and s == args.steps - 1)
            wall += d
            solve += s_ms
            its += t
            pm += a
            pl += b_
        barrier()
        clocks = sampler.stop()
        launches = ctx.launches - l0
        wall_max, solve_max, pm_max = reduce_max([wall, solve, pm])
        launches_all, = reduce_sum([float(launches)])
        if rank == 0 and args.dump_outputs:  # rank 0's results: W holds rows [0, r1) of the global W, the rest is replicated
            dump_outputs(args.dump_outputs, {name: st[name] for name in BATCH_FIELDS})
        if rank == 0:
            nloc = r1 - r0
            achieved = 4.0 * nloc * m * k * R * pl / (pm_max * 1e-3) / 1e12 if pm_max > 0 else float("nan")
            line = {
                "metric": METRIC, "value": its / (solve_max * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": solve_max / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOADS["C5"] % iters, "rows_per_gpu": nloc,
                           "engine": "tiled, row-sharded: tcgen05 pass per GPU + one NCCL all-reduce of the k x m x R numerators "
                                     "and colsum(W) per iteration", "l2": "inputs larger than L2 (%.1f GB of X per GPU)" % (nloc * m * 4 / 1e9),
                           "restart_iterations_per_step": its / args.steps, "same_config": True},
                "clocks": clocks,
                "e2e": {"value": its / wall_max, "unit": UNIT, "h2d_bytes_per_step": nloc * m * 4, "d2h_bytes_per_step": R * 4 * 8,
                        "ms_per_step": wall_max / args.steps * 1e3,
                        "call": "nmfk_set_X (H2D of this rank's rows) + device Philox factors + nmfk_solve + state read-back"},
                "gpu_launches": int(launches_all),
                "roofline": {"bound": "tensor", "achieved": achieved, "peak": tf32 / 3.0, "unit": "TFLOP/s",
                             "frac": achieved / (tf32 / 3.0), "traffic": None,
                             "kernel": "tc_pass_kernel (per GPU; one launch = one half-update of all 32 restarts on this GPU's rows)",
                             "launch_ms": pm_max / max(pl, 1), "launches_timed": int(pl),
                             "peak_source": "tcgen05 kind::tf32 dense (nmfk_measure_peak 13: %.1f TFLOP/s) / 3" % tf32}}

    elif cfg == "C2":
        if world != 1:
            raise SystemExit("bench.py: --config C2 runs on one GPU")
        r = bench_c2(ctx, nb, synth, torch, args, flush, args.steps, args.warmup, dump=args.dump_outputs)
        line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": {"workload": WORKLOADS["C2"], "kopt": r["kopt"], "same_config": True,
                                                "l2": "256 MiB written between steps (X itself is 1.6 MB and L2-resident by design)"},
                "e2e": {"value": r["restart_iterations_per_step"] / r["e2e_s_execute"], "unit": UNIT,
                        "h2d_bytes_per_step": 1000 * 200 * 8, "d2h_bytes_per_step": sum((1000 * k + k * 200) * 8 for k in range(2, 11))},
                "gpu_launches": int(ctx.launches), "roofline": dict(r["roofline"], traffic=TRAFFIC["C2"][0])}
        if not args.no_cpu_baseline:
            threads = pin_blas()
            t, d, what = cpu_step("C2", 0)
            line["cpu_baseline"] = {"value": t / d, "unit": UNIT, "cores": threads, "kind": "port", "sample": what}

    if rank == 0 and line is not None:
        print(json.dumps(line))
    ctx.close()
    if use_dist:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
