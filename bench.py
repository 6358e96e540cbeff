#!/usr/bin/env python
"""bench.py -- QPALM hot path on B200: batched QP solves/sec and dense-QP time-to-solution.

Contract (driver):  python bench.py --gpus N --steps K --warmup W [--impl reference]
For N > 1 the driver launches one rank per GPU with torch.distributed.run; the ranks shard the
independent QPs with no data-path collective (weak scaling: instances per GPU fixed).

A *step* is one pass of the hot path over one batch of synthetic QPs:
  workload "mpc_batch"  (BASELINE config 4): `--batch` chain80w-sized QPs (n=240, m=949, shared Q/A) per GPU,
                        every QP solved from a cold start to eps 1e-6 through the batch entry point.
  workload "dense"      (BASELINE config 3): one dense QP n=8000, m=16000 solved to eps 1e-6 (time-to-solution),
                        reported as the `time_to_solution` block of the same JSON line at N = 1 and as the
                        primary line when the batch kernels are not built.
`value` is whole-job throughput with all inputs resident in HBM (CUDA-event time on the launching stream, max over
ranks); `e2e` goes through the public C API with host buffers (setup/H2D + solve + D2H inside the timed region).
`--dump-outputs DIR` writes, after the timed steps, what the last step computed (rank 0's x, y and info fields per QP) as
DIR/<name>.npy, so that two builds can be compared output for output: the inputs are seeded, the same arguments give the
same inputs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from qpalm_b200 import abi, problems  # noqa: E402
from qpalm_b200.interface import Qpalm, load_library  # noqa: E402


# ------------------------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def product_lib():
    lib = load_library("b200")
    lib.qpalm_b200_get_stats.argtypes = [C.POINTER(abi.QPALMWorkspace), C.POINTER(abi.QPALMB200Stats)]
    lib.qpalm_b200_bench_dmma_peak.argtypes = [C.POINTER(C.c_double)]
    lib.qpalm_b200_bench_gemv.argtypes = [abi.c_int, abi.c_int, abi.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.qpalm_b200_bench_dsyrk.argtypes = [abi.c_int, abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    lib.qpalm_b200_bench_potrf.argtypes = [abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    return lib


def get_stats(lib, solver) -> abi.QPALMB200Stats:
    st = abi.QPALMB200Stats()
    lib.qpalm_b200_get_stats(solver._work, C.byref(st))
    return st


DUMP_BYTES = 60_000_000     # --dump-outputs: data bytes in all (64 MB less room for the .npy headers)


def solve_outputs(prefix, x, y, infos):
    """What a caller of the timed path receives: x, y and the info fields, one row per QP."""
    out = {prefix + "x": x, prefix + "y": y}
    out.update({prefix + k: [i[k] for i in infos] for k in ("status_val", "iter", "iter_out", "objective")})
    return out


def dump_outputs(out_dir, outputs):
    """Every array of `outputs` as <out_dir>/<name>.npy in float64.  When they come to more than DUMP_BYTES, every array
    keeps the same fixed, seeded fraction of its rows (axis 0), whose indices go to <name>_rows.npy."""
    arrays = {k: np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in outputs.items()}
    data = sum(a.nbytes for a in arrays.values())
    with_rows = data + sum(8 * len(a) for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if data > DUMP_BYTES:
            rows = np.sort(np.random.default_rng(0).choice(len(a), max(1, len(a) * DUMP_BYTES // with_rows), replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------
# reference / oracle CPU arm
# ------------------------------------------------------------------------------------------------------
def cpu_impl():
    from oracle import refbind   # the checker libraries: cpu_baseline / --impl reference legs only
    return ("reference", "reference") if refbind.have_reference() else ("oracle", "port")


def cpu_threads():
    return os.cpu_count() or 1


def run_cpu_dense_sample(n, m, seed):
    """Reference CPU path on a bounded sample of the dense workload: same generator, n x m reduced so that one
    solve is ~10-30 s of CPU work.  Returns (seconds per solve, iterations)."""
    impl, kind = cpu_impl()
    os.environ.setdefault("OPENBLAS_NUM_THREADS", str(cpu_threads()))
    from oracle import refbind
    refbind.interface.load_library(impl)
    refbind.set_blas_threads(cpu_threads())
    p = problems.dense_qp(n, m, seed=seed)
    s = Qpalm(impl)
    for k, v in p.settings.items():
        setattr(s.settings, k, v)
    s.set_data(p.Q, p.A, p.q, p.bmin, p.bmax)
    t0 = time.perf_counter()
    s._allocate_work()
    s._solve()
    dt = time.perf_counter() - t0
    r = s.result()
    s.cleanup()
    return dt, r, kind


class CpuBatchPool:
    """The reference CPU path for the batch workload: one single-threaded reference process per host core over disjoint
    instance ranges (QPALM is single-threaded).  The worker pool is created -- and the reference library loaded in the
    parent, so the driver's loaded-library hook sees it -- BEFORE any timed region.

    mode "setup_per_instance":  qpalm_setup + qpalm_solve + qpalm_cleanup per instance (what a naive caller does).
    mode "update_per_instance": ONE qpalm_setup per worker, then qpalm_update_q + qpalm_update_bounds + qpalm_solve per
                                instance (src/qpalm.c:793-871) -- the cheaper way to drive the reference over a sweep
                                that shares Q and A, i.e. the fairer baseline for the batch engine."""

    def __init__(self, b, cores=None):
        import multiprocessing as mp
        from oracle import refbind   # cpu_baseline / --impl reference legs only
        self.impl, self.kind = cpu_impl()
        interface_lib = refbind.interface.load_library(self.impl)      # noqa: F841  loaded in the parent, inherited by fork
        self.cores = cores or cpu_threads()
        global _CPU_BATCH
        _CPU_BATCH = b          # inherited by the forked workers (ctypes-backed matrices cannot be pickled)
        self.pool = mp.get_context("fork").Pool(self.cores)
        self.pool.map(_cpu_batch_warm, [self.impl] * self.cores)

    def run(self, count, mode="setup_per_instance", first=0):
        """Timed: `count` instances starting at `first`.  Returns (solves/sec, per-instance iterations, per-instance x)."""
        cores = min(self.cores, count)
        chunks = [list(range(first + k, first + count, cores)) for k in range(cores)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_batch_worker, [(self.impl, ch, mode) for ch in chunks])
        dt = time.perf_counter() - t0
        its, xs = {}, {}
        for r in res:
            for k, it, x in r:
                its[k], xs[k] = it, x
        order = sorted(its)
        return count / dt, [its[k] for k in order], [xs[k] for k in order]

    def close(self):
        self.pool.close()
        self.pool.join()


_CPU_BATCH = None


def _cpu_batch_warm(impl):
    from oracle import refbind
    refbind.interface.load_library(impl)
    refbind.set_blas_threads(1)      # one single-threaded reference process per core
    return os.getpid()


def _cpu_batch_worker(arg):
    impl, idx, mode = arg
    b = _CPU_BATCH
    from oracle.refbind import Qpalm as RefQpalm, solve_qp
    out = []
    if mode == "update_per_instance" and idx:
        q0 = b.instance(idx[0])
        s = RefQpalm(impl)
        for k, v in q0.settings.items():
            setattr(s.settings, k, v)
        s.set_data(q0.Q, q0.A, q0.q, q0.bmin, q0.bmax)
        assert s._allocate_work()
        for j, k in enumerate(idx):
            if j:
                s._update_q(b.q[k])
                s._update_bounds(b.bmin[k], b.bmax[k])
                s._warm_start(np.zeros(q0.n), np.zeros(q0.m))     # cold start, as the batch engine does
            s._solve()
            r = s.result()
            out.append((k, r.iter, r.x))
        s.cleanup()
        return out
    for k in idx:
        q = b.instance(k)
        r = solve_qp(impl, q.Q, q.A, q.q, q.bmin, q.bmax, **q.settings)
        out.append((k, r.iter, r.x))
    return out


def committed_reference(name):
    """Reference record generated ONCE in the build container at the BASELINE size (tests/golden/make_golden_big.py)."""
    path = os.path.join(ROOT, "tests", "golden", name + ".json")
    if not os.path.exists(path):
        return None
    d = json.load(open(path))
    return {k: d.get(k) for k in ("case", "status_val", "iter", "iter_out", "objective", "setup_seconds_wall", "solve_seconds_wall",
                                  "host_cores", "blas_threads", "host", "reference", "input_sha256")}


# ------------------------------------------------------------------------------------------------------
# dense workload (BASELINE config 3)
# ------------------------------------------------------------------------------------------------------
def bench_dense(args, lib, steps, warmup, sample_clocks=True):
    import torch
    n, m = args.n, args.m
    p = problems.dense_qp(n, m, seed=args.seed)
    h2d = 8 * (p.A.x.size + p.Q.x.size + n + 2 * m)
    d2h = 8 * (n + m)
    s = Qpalm("b200")
    for k, v in p.settings.items():
        setattr(s.settings, k, v)
    s.set_data(p.Q, p.A, p.q, p.bmin, p.bmax)
    t0 = time.perf_counter()
    assert s._allocate_work(), "qpalm_setup failed"
    setup_s = time.perf_counter() - t0
    for _ in range(warmup):
        s._solve()
    st0 = get_stats(lib, s)
    sampler = ClockSampler(torch.cuda.current_device())
    if sample_clocks:
        sampler.start()
    torch.cuda.synchronize()
    for _ in range(steps):
        s._solve()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sample_clocks else None
    st1 = get_stats(lib, s)
    res = s.result()
    dev_ms = st1.device_ms_total - st0.device_ms_total
    out = dict(
        ms_per_solve=dev_ms / steps, status=res.status, iter=res.iter, iter_out=res.iter_out, setup_s=setup_s,
        launches=int(st1.kernel_launches - st0.kernel_launches),
        refactorizations=int(st1.refactorizations - st0.refactorizations) // steps,
        refactor_active_avg=(st1.refactor_active_sum - st0.refactor_active_sum) / max(1, st1.refactorizations - st0.refactorizations),
        updown_sweeps=int(st1.updown_calls - st0.updown_calls) // steps,
        ms_factor=(st1.device_ms_factor - st0.device_ms_factor) / steps,
        ms_updown=(st1.device_ms_updown - st0.device_ms_updown) / steps,
        dense_flops=(st1.dense_flops - st0.dense_flops) / steps,
        factor_flops_executed=((st1.dense_flops - st0.dense_flops) - 2.0 * float(n) * n * ((st1.updown_rank_sum - st0.updown_rank_sum)
                               + (st1.inner_iterations - st0.inner_iterations))) / steps,      # minus update sweeps (2 k n^2) and solves (2 n^2)
        updown_rank_sum=int(st1.updown_rank_sum - st0.updown_rank_sum) // steps,
        sigma_update_calls=int(st1.sigma_update_calls - st0.sigma_update_calls) // steps, alg_bytes=(st1.algorithmic_bytes - st0.algorithmic_bytes) / steps,
        clocks=clocks, h2d=h2d, d2h=d2h, x=res.x, y=res.y, objective=res.objective, status_val=res.status_val)
    s.cleanup()
    # e2e: setup (H2D + Ruiz) + solve + solution read-back through the public API, host buffers (pageable, as the caller's CSC
    # arrays are; pinning the 1.28 GB of matrix values made qpalm_setup slower on the box: 0.63 s against 0.21 s)
    e2e, setup_warm = [], []
    for _ in range(max(1, min(steps, 2))):
        t0 = time.perf_counter()
        s2 = Qpalm("b200")
        for k, v in p.settings.items():
            setattr(s2.settings, k, v)
        s2.set_data(p.Q, p.A, p.q, p.bmin, p.bmax)
        s2._allocate_work()
        setup_warm.append(time.perf_counter() - t0)
        s2._solve()
        r2 = s2.result()
        e2e.append(time.perf_counter() - t0)
        s2.cleanup()
        assert r2.status_val == res.status_val
    out["e2e_s"] = float(np.mean(e2e))
    out["setup_warm_s"] = float(np.mean(setup_warm))   # setup_s above is the first call of the process (CUDA context + module load)
    return out, p


def dense_reference_block(args, dense, p):
    """The committed reference record of this exact problem (tests/golden/, generated once on the build container's host cores)
    next to the GPU time, and the parity of THIS run's solution against it (north-star gates: status, x / y 1e-8, iterations 5 %)."""
    if (args.n, args.m, args.seed) != (8000, 16000, 0):
        return None
    name = "c3_dense_n8000_m16000_s0"
    rec = committed_reference(name)
    if rec is None:
        return {"unavailable": f"tests/golden/{name}.json not committed"}
    import hashlib
    h = hashlib.sha256()
    for a in (p.Q.p, p.Q.i, p.Q.x, p.A.p, p.A.i, p.A.x, p.q, p.bmin, p.bmax):
        h.update(np.ascontiguousarray(a).tobytes())
    out = {"label": "COMMITTED reference run (unmodified reference, CHOLMOD build), not timed in this process",
           "setup_seconds": rec["setup_seconds_wall"], "solve_seconds": rec["solve_seconds_wall"], "host_cores": rec["host_cores"],
           "blas_threads": rec["blas_threads"], "host": rec["host"], "status_val": rec["status_val"], "iter": rec["iter"],
           "iter_out": rec["iter_out"], "same_input_bytes": h.hexdigest() == rec["input_sha256"]}
    npz = os.path.join(ROOT, "tests", "golden", name + ".npz")
    if out["same_input_bytes"] and os.path.exists(npz):
        g = np.load(npz)
        rel = lambda a, b: float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))
        out["parity"] = {"x_rel_error": rel(dense["x"], g["x"]), "y_rel_error": rel(dense["y"], g["y"]),
                         "iter_gpu": dense["iter"], "iter_ref": rec["iter"], "iter_out_gpu": dense["iter_out"], "iter_out_ref": rec["iter_out"],
                         "objective_gpu": dense["objective"], "objective_ref": rec["objective"]}
    out["gpu_solve_seconds"] = dense["ms_per_solve"] * 1e-3
    out["gpu_setup_plus_solve_seconds"] = dense["e2e_s"]
    out["ratio_solve"] = rec["solve_seconds_wall"] / (dense["ms_per_solve"] * 1e-3)
    out["ratio_setup_plus_solve"] = (rec["setup_seconds_wall"] + rec["solve_seconds_wall"]) / dense["e2e_s"]
    return out


def tensor_roofline(lib, n, k_avg, dense):
    """Dominant kernel of the dense workload: k_dgemm_nt (FP64 DMMA).  achieved = algorithmic flops of the
    refactorisations (n^2 |J| SYRK + n^3/3 Cholesky, SURVEY 8(d)) / their CUDA-event time inside the timed solves."""
    peak = C.c_double(0)
    lib.qpalm_b200_bench_dmma_peak(C.byref(peak))
    # SURVEY 8(d) model: every refactorisation re-forms A_J' Sigma A_J (n^2 |J|) and factors (n^3 / 3).  EXECUTED: H is kept and
    # updated incrementally (n^2 |Delta| per refactorisation), so the flops the kernels really ran are fewer; `frac` uses those.
    flops_model = dense["refactorizations"] * (float(n) * n * k_avg + float(n) ** 3 / 3.0)
    flops = dense["factor_flops_executed"]
    ach = flops / max(dense["ms_factor"], 1e-9) / 1e9     # TFLOP/s
    ach_model = flops_model / max(dense["ms_factor"], 1e-9) / 1e9
    ms = C.c_double(0)
    lib.qpalm_b200_bench_dsyrk(n, max(16, int(k_avg)), 3, C.byref(ms))
    syrk_tf = float(n) * n * max(16, int(k_avg)) / max(ms.value, 1e-9) / 1e9
    lib.qpalm_b200_bench_potrf(n, 2, C.byref(ms))
    potrf_tf = float(n) ** 3 / 3 / max(ms.value, 1e-9) / 1e9
    return {"bound": "tensor", "achieved": ach, "peak": peak.value, "unit": "TFLOP/s", "frac": ach / max(peak.value, 1e-9),
            "traffic": None, "kernel": "k_dgemm_nt (FP64 DMMA SYRK + Cholesky trailing updates)",
            "flops": "executed (incremental n^2 |Delta| SYRK + n^3/3 per refactorisation) / CUDA-event time of the refactorisations",
            "model_8d": {"achieved": ach_model, "frac": ach_model / max(peak.value, 1e-9),
                         "note": "SURVEY 8(d) per-refactorisation model n^2 |J| + n^3/3 over the same time (counts flops the incremental H update never executes)"},
            "peak_source": "in-repo mma.sync.m8n8k4.f64 issue-rate microbenchmark (MEASURED_PEAKS.json has no FP64 entry)",
            "syrk_alone_tflops": syrk_tf, "potrf_alone_tflops": potrf_tf}


def sparse_spmv_roofline(lib, hbm):
    """Q x, A x, A' y over CSR / CSC (k_csr_spmv: a warp per row / column, 128-bit value + 64-bit index loads) at the C1 and
    C2 shapes of BASELINE.json.  bytes = 12 nnz + 4 (rows + 1) + 8 (rows + cols) per product (SURVEY 8(d) storage model)."""
    lib.qpalm_b200_bench_spmv.argtypes = [C.POINTER(abi.SolverSparse), C.POINTER(abi.SolverSparse), abi.c_int, C.POINTER(C.c_double),
                                          C.POINTER(abi.c_int)]
    out = {}
    shapes = {"C1 random sparse n=1000 m=2000 density 0.05": lambda: problems.random_qp(1000, 2000, 0.05, 0.007, seed=1),
              "C2 stand-in (SYNTHETIC grid QP, CONT-300 class) n=90000 m=359102": lambda: problems.grid_qp(300, seed=0)}
    for name, make in shapes.items():
        p = make()
        ms, nnz = (C.c_double * 3)(), (abi.c_int * 3)()
        rc = lib.qpalm_b200_bench_spmv(p.A.ptr(), p.Q.ptr(), 50, ms, nnz)
        if rc:
            out[name] = {"unavailable": f"qpalm_b200_bench_spmv rc {rc}"}
            continue
        n, m = p.n, p.m
        dims = {"A_times_x": (m, n), "At_times_y": (n, m), "Q_times_x": (n, n)}
        blk = {}
        for k, key in enumerate(dims):
            rows, cols = dims[key]
            by = 12.0 * nnz[k] + 4.0 * (rows + 1) + 8.0 * (rows + cols)
            gbs = by / (ms[k] * 1e-3) / 1e9
            blk[key] = {"achieved": gbs, "frac": gbs / hbm, "us": 1e3 * ms[k], "nnz": int(nnz[k]), "bytes": by}
        blk["note"] = ("working set %.1f MB: L2-resident after the first touch (126 MB L2), so this is launch latency + L2 bandwidth, not HBM"
                       % ((12.0 * (nnz[0] + nnz[2])) / 1e6)) if 12.0 * (nnz[0] + nnz[2]) < 100e6 else "working set exceeds L2"
        out[name] = blk
    return out


def hbm_roofline(lib, n, m):
    hbm, src = measured_peaks()
    a, b = C.c_double(0), C.c_double(0)
    lib.qpalm_b200_bench_gemv(n, m, 20, C.byref(a), C.byref(b))
    bytes_ = 8.0 * n * m
    out = {"bound": "hbm", "unit": "GB/s", "peak": hbm, "peak_source": src,
           "A_times_x": {"achieved": bytes_ / (a.value * 1e-3) / 1e9, "frac": bytes_ / (a.value * 1e-3) / 1e9 / hbm},
           "At_times_y": {"achieved": bytes_ / (b.value * 1e-3) / 1e9, "frac": bytes_ / (b.value * 1e-3) / 1e9 / hbm}}
    try:
        out["sparse"] = sparse_spmv_roofline(lib, hbm)
    except Exception as ex:      # never lose the bench line over a side measurement
        out["sparse"] = {"unavailable": repr(ex)}
    return out


# ------------------------------------------------------------------------------------------------------
# batched MPC workload (BASELINE config 4)
# ------------------------------------------------------------------------------------------------------
# dominant kernel per batch engine (share of the step from the ncu launch lists under profiles/): the persistent engine IS
# one kernel; in the lock-step engine the single-CTA diagonal-block factorisation leads (39 %)
DOMINANT_KERNEL = {"persistent": "kbp_solve", "lockstep": "k_diag_block"}
def ncu_traffic(kernel, nb):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, read from profiles/ncu_traffic.json --
    written by tools/ncu_full_summary.py from the `ncu --set full` capture of this command, together with the capture's file
    name and the batch size it was taken at.  null when no capture matches the batch size being benchmarked."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, None
    for ent in json.load(open(path)).get(kernel, []):
        if int(ent.get("batch", -1)) == int(nb):
            return float(ent["dram_bytes"]), ent.get("source")
    return None, None


def batch_algorithmic_bytes(n, m, stats):
    """SURVEY.md 8(d) byte model (dense storage), summed over the steps the instances actually executed:
    per inner iteration 2 B_A + B_Q + 8(38m + 26n) + 2 B_L (solve); per outer iteration 8(7m + 4n);
    per refactorisation 8 |J| n + 2 B_L.  B_A = 8mn, B_Q = B_L = 8 n(n+1)/2."""
    BA, BQ = 8.0 * m * n, 8.0 * n * (n + 1) / 2
    BL = BQ
    return (stats["inner"] * (2 * BA + BQ + 8.0 * (38 * m + 26 * n) + 2 * BL) + stats["outer"] * 8.0 * (7 * m + 4 * n)
            + stats["refactorizations"] * 2 * BL + 8.0 * n * stats["refactor_J_sum"])


def batch_roofline(n, m, nb, r, steps):
    hbm, src = measured_peaks()
    k = [v for name, v in r["kprof"].items() if r["dominant"] in name]
    launches = sum(v["launches"] for v in k)
    ms = sum(v["ms"] for v in k)
    if not launches:
        return None
    per_launch_ms = ms / launches
    if r["dominant"] == "kbp_solve":       # one launch = the whole sweep of nb instances
        bytes_per_launch = batch_algorithmic_bytes(n, m, r["stats"])
        note = "one launch solves the whole batch; bytes = SURVEY 8(d) model over the executed iterations (shared A, Q counted per instance)"
    else:                                  # k_diag_block: read + write one 128 x 128 lower block, write its inverse, per instance
        bytes_per_launch = nb * 3 * 8.0 * 128 * 129 / 2
        note = "per launch: every instance's 128 x 128 diagonal block read + written, inverse written (upper bound: masked instances skip)"
    ach = bytes_per_launch / (per_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(r["dominant"], nb)
    return {"bound": "hbm", "kernel": r["dominant"], "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": src, "launches_timed": launches, "ms_per_launch": per_launch_ms, "share_of_step": ms / max(r["dev_ms"], 1e-9),
            "algorithmic_bytes_per_launch": bytes_per_launch, "note": note}


def bench_batch(args, steps, warmup, rank, world):
    import torch
    from qpalm_b200 import batch as qb
    nb = args.batch
    b = problems.mpc_batch(nb, seed=args.seed + 1000 * rank)     # each rank owns a disjoint set of instances
    h = qb.Batch(b.Q, b.A, b.settings, nb)
    assert h.ok, "batch setup failed"
    h.upload(b.q, b.bmin, b.bmax)
    for _ in range(warmup):
        h.solve_resident(nb)
    engine = h.stats(nb)["engine"]
    dominant = DOMINANT_KERNEL[engine]
    lib = h.lib
    lib.qpalm_b200_prof_enable.argtypes = [C.c_char_p]
    lib.qpalm_b200_prof_report.argtypes = [C.c_char_p, C.c_size_t]
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    lib.qpalm_b200_prof_enable(dominant.encode())     # CUDA-event pair around every launch of the dominant kernel only
    dev_ms = 0.0
    for _ in range(steps):
        dev_ms += h.solve_resident(nb)
    torch.cuda.synchronize()
    buf = C.create_string_buffer(1 << 16)
    lib.qpalm_b200_prof_report(buf, len(buf))
    lib.qpalm_b200_prof_enable(b"")
    kprof = json.loads(buf.value.decode() or "{}")
    clocks = sampler.stop()
    x, y, infos = h.download(nb)
    stats = h.stats(nb)
    # e2e: host buffers in, host results out, every step
    if world > 1:
        torch.distributed.barrier()
    # inputs and results in PINNED host memory (the buffers a caller that cares about transfer time hands to the C entry point)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).pin_memory().numpy()
    qh, bminh, bmaxh = pin(b.q), pin(b.bmin), pin(b.bmax)
    xh, yh = pin(np.zeros_like(x)), pin(np.zeros_like(y))
    from qpalm_b200.abi import QPALMInfo
    ih = (QPALMInfo * nb)()
    h.solve(qh, bminh, bmaxh, x=xh, y=yh, info=ih, raw_info=True)     # untimed: first-touch of the result buffers
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        xe, ye, ie = h.solve(qh, bminh, bmaxh, x=xh, y=yh, info=ih, raw_info=True)
    e2e_s = (time.perf_counter() - t0) / steps
    assert all(int(ie[k].status_val) == infos[k]["status_val"] for k in range(nb)) and np.array_equal(xe, x), "e2e results differ from the resident run"
    launches = h.last_launches() if hasattr(h, "last_launches") else None
    h.cleanup()
    return dict(dev_ms=dev_ms, e2e_s=e2e_s, clocks=clocks, infos=infos, x=x, y=y, b=b, launches=launches, stats=stats, kprof=kprof,
                dominant=dominant,
                h2d=8 * (b.q.size + b.bmin.size + b.bmax.size), d2h=8 * (x.size + y.size))


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "dense", "mpc_batch"])
    ap.add_argument("--n", type=int, default=8000)
    ap.add_argument("--m", type=int, default=16000)
    ap.add_argument("--batch", type=int, default=512, help="instances per GPU (4096 / 8)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-n", type=int, default=1600, help="dense CPU sample size (m = 2n)")
    ap.add_argument("--cpu-batch", type=int, default=0, help="batch CPU sample size (0: one instance per host core)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense time-to-solution block")
    ap.add_argument("--sweep-total", type=int, default=4096, help="N = 1: also run the whole sweep on the one GPU (0 to skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    rank, world, local = dist_env()
    steps, warmup = max(1, args.steps), max(3, args.warmup) if args.impl == "b200" else max(0, args.warmup)

    # ---------------- reference arm: the reference's CPU implementation, bounded sample ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        workload = args.workload
        if workload == "auto":
            workload = "mpc_batch"
        impl, kind = cpu_impl()
        if workload == "dense":
            vals = []
            for _ in range(steps):
                dt, r, kind = run_cpu_dense_sample(args.cpu_n, 2 * args.cpu_n, args.seed)
                vals.append(dt)
            v = 1.0 / float(np.mean(vals))
            sample = f"same generator at n={args.cpu_n}, m={2 * args.cpu_n} (setup+solve), {cpu_threads()} BLAS threads"
            cfg = {"workload": f"dense random convex QP n={args.n} m={args.m} eps 1e-6", "sample": sample}
            line = {"metric": "qp_solves_per_sec", "value": v, "unit": "solves/s", "ms_per_step": 1e3 / v}
            cores = cpu_threads()
        else:
            b = problems.mpc_batch(args.batch, seed=args.seed)
            count = args.cpu_batch or min(args.batch, 2 * cpu_threads())
            pool = CpuBatchPool(b)          # workers forked and the reference library loaded BEFORE the timed steps
            kind, cores = pool.kind, min(pool.cores, count)
            for _ in range(max(0, args.warmup > 0)):
                pool.run(min(count, cpu_threads()))
            vals, vals_upd = [], []
            for _ in range(steps):
                vals.append(pool.run(count, "setup_per_instance")[0])
            for _ in range(steps):
                vals_upd.append(pool.run(count, "update_per_instance")[0])
            pool.close()
            v, v_upd = float(np.mean(vals)), float(np.mean(vals_upd))
            sample = f"{count} of the {args.batch} instances per step, one single-threaded reference process per host core ({cores})"
            cfg = {"workload": f"batched MPC sweep: {args.batch} chain80w-sized QPs (n=240, m=949) per GPU, eps 1e-6", "sample": sample,
                   "value_is": "the FASTER of the two ways of driving the reference over the sweep",
                   "setup_per_instance_solves_per_sec": v, "update_per_instance_solves_per_sec": v_upd,
                   "update_per_instance": "one qpalm_setup per worker, then qpalm_update_q + qpalm_update_bounds + cold qpalm_solve per instance"}
            v = max(v, v_upd)
            line = {"metric": "qp_solves_per_sec", "value": v, "unit": "solves/s", "ms_per_step": 1e3 * count / v}
        line.update({"impl": "reference", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "higher_is_better": True,
                     "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                     "cpu_baseline": {"value": line["value"], "unit": "solves/s", "cores": cores, "kind": kind, "sample": sample},
                     "e2e": {"value": line["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        print(json.dumps(line))
        return

    # ---------------- product arm ----------------
    import torch
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product has no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = product_lib()
    from qpalm_b200 import batch as qb
    workload = args.workload
    if workload == "auto":
        workload = "mpc_batch" if qb.available() else "dense"

    line = {"n_gpus": world, "steps": steps, "warmup": warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic"}
    if workload == "mpc_batch":
        r = bench_batch(args, steps, warmup, rank, world)
        outputs = solve_outputs("", r["x"], r["y"], r["infos"])
        t = torch.tensor([r["dev_ms"], r["e2e_s"]], device="cuda", dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        dev_ms, e2e_s = float(t[0]), float(t[1])
        total = args.batch * world
        solved = sum(1 for i in r["infos"] if i["status_val"] == 1)
        line.update({"metric": "qp_solves_per_sec", "unit": "solves/s", "value": total * steps / (dev_ms * 1e-3),
                     "ms_per_step": dev_ms / steps,
                     "config": {"workload": f"batched MPC sweep: {args.batch} chain80w-sized QPs (n=240, m=949, shared Q/A) per GPU, "
                                            f"cold start, eps 1e-6; {total} QPs in flight over {world} GPU(s)",
                                "batch_per_gpu": args.batch, "l2": "working set (per-instance factors) larger than L2",
                                "solved": f"{solved}/{args.batch} on rank 0"},
                     "e2e": {"value": total / e2e_s, "unit": "solves/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"]},
                     "clocks": r["clocks"], "gpu_launches": r["launches"]})
        if rank == 0:
            iters = float(np.mean([i["iter"] for i in r["infos"]]))
            line["config"]["mean_iterations"] = iters
            line["config"]["engine"] = r["stats"]["engine"]
            b0 = r["b"]
            line["roofline"] = batch_roofline(b0.q.shape[1], b0.bmin.shape[1], args.batch, r, steps)
            if not args.no_cpu and world == 1:      # the CPU baseline is reported at N = 1 only
                b = r["b"]
                count = args.cpu_batch or min(args.batch, 2 * cpu_threads())
                pool = CpuBatchPool(b)
                v, cpu_iters, cpu_x = pool.run(count, "setup_per_instance")
                v_upd = pool.run(count, "update_per_instance")[0]
                pool.close()
                line["cpu_baseline"] = {"value": max(v, v_upd), "unit": "solves/s", "cores": min(pool.cores, count), "kind": pool.kind,
                                        "sample": f"first {count} instances of rank 0's batch, one single-threaded reference process per core "
                                                  f"(pool created before timing); setup per instance {v:.1f} solves/s, one setup per worker + "
                                                  f"update_q / update_bounds per instance {v_upd:.1f} solves/s"}
                # per-instance parity of the SAME instances: GPU batch engine vs the reference (north-star gates)
                gi = [i["iter"] for i in r["infos"][:count]]
                relx = [float(np.max(np.abs(r["x"][k] - cpu_x[k])) / max(1.0, float(np.max(np.abs(cpu_x[k]))))) for k in range(count)]
                line["config"]["parity_sample"] = {"instances": count, "max_rel_x_error": max(relx),
                                                   "max_iteration_difference": int(max(abs(a - c) for a, c in zip(gi, cpu_iters))),
                                                   "gpu_mean_iterations": float(np.mean(gi)), "reference_mean_iterations": float(np.mean(cpu_iters)),
                                                   "gates": "x within 1e-8 relative, iterations within 5 %"}
    else:
        if world > 1:   # BASELINE config 3 on N GPUs: ONE QP, constraint rows sharded over the ranks (csrc/shard.cu, NCCL)
            from qpalm_b200 import rowshard
            rowshard.init(rank, world, torch.device("cuda", local))
            line["scaling"] = "strong"
        dense, p = bench_dense(args, lib, steps, warmup)
        outputs = solve_outputs("", dense["x"], dense["y"], [dense])
        t = torch.tensor([dense["ms_per_solve"], dense["e2e_s"]], device="cuda", dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            dense["ms_per_solve"], dense["e2e_s"] = float(t[0]), float(t[1])
        dev_ms = dense["ms_per_solve"]
        line.update({"metric": "qp_solves_per_sec", "unit": "solves/s", "value": 1e3 / dev_ms, "ms_per_step": dev_ms,
                     "config": {"workload": f"dense random convex QP n={args.n} m={args.m} eps 1e-6"
                                            + (f" (constraint rows sharded over {world} GPUs, NCCL)" if world > 1 else ""),
                                "l2": "inputs larger than L2 (A' is %.2f GB)" % (8.0 * args.n * args.m / 1e9),
                                "status": dense["status"], "iter": dense["iter"], "iter_out": dense["iter_out"]},
                     "e2e": {"value": 1.0 / dense["e2e_s"], "unit": "solves/s", "h2d_bytes_per_step": dense["h2d"], "d2h_bytes_per_step": dense["d2h"]},
                     "clocks": dense["clocks"], "gpu_launches": dense["launches"] // steps})
        if rank == 0:
            line["roofline"] = tensor_roofline(lib, args.n, dense["refactor_active_avg"], dense)
            line["roofline_hbm"] = hbm_roofline(lib, args.n, args.m)
            line["time_to_solution"] = {"seconds": dev_ms * 1e-3, "e2e_seconds": dense["e2e_s"], "setup_seconds": dense["setup_warm_s"], "setup_seconds_first_call": dense["setup_s"],
                                        "refactorizations": dense["refactorizations"], "updown_sweeps": dense["updown_sweeps"],
                                        "updown_rank_sum": dense["updown_rank_sum"], "sigma_update_calls": dense["sigma_update_calls"],
                                        "ms_in_refactorizations": dense["ms_factor"], "ms_in_updown": dense["ms_updown"]}
            if world == 1:
                line["time_to_solution"]["reference"] = dense_reference_block(args, dense, p)
            if not args.no_cpu and world == 1:
                dt, rr, kind = run_cpu_dense_sample(args.cpu_n, 2 * args.cpu_n, args.seed)
                line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "solves/s", "cores": cpu_threads(), "kind": kind,
                                        "sample": f"same generator at n={args.cpu_n}, m={2 * args.cpu_n} (setup+solve {dt:.2f} s, "
                                                  f"{rr.iter} iterations); Newton-system flops scale ~ (n/{args.cpu_n})^3"}
    # the dense time-to-solution block rides along on the batch line at N = 1
    if workload == "mpc_batch" and world == 1 and not args.no_dense:
        dense, p = bench_dense(args, lib, 1, 1, sample_clocks=False)
        outputs.update(solve_outputs("dense_", dense["x"], dense["y"], [dense]))
        line["time_to_solution"] = {"workload": f"dense random convex QP n={args.n} m={args.m} eps 1e-6",
                                    "seconds": dense["ms_per_solve"] * 1e-3, "e2e_seconds": dense["e2e_s"], "setup_seconds": dense["setup_warm_s"], "setup_seconds_first_call": dense["setup_s"],
                                    "status": dense["status"], "iter": dense["iter"], "iter_out": dense["iter_out"],
                                    "refactorizations": dense["refactorizations"], "ms_in_refactorizations": dense["ms_factor"],
                                    "updown_sweeps": dense["updown_sweeps"], "updown_rank_sum": dense["updown_rank_sum"],
                                    "sigma_update_calls": dense["sigma_update_calls"], "ms_in_updown": dense["ms_updown"],
                                    "reference": dense_reference_block(args, dense, p)}
        line["roofline_tensor"] = tensor_roofline(lib, args.n, dense["refactor_active_avg"], dense)
        line["roofline_hbm"] = hbm_roofline(lib, args.n, args.m)
    if workload == "mpc_batch" and world == 1 and not args.no_dense and args.sweep_total > args.batch:
        # the WHOLE sweep (BASELINE config 4: 4096 instances) on ONE GPU, several waves through the engine's work queue:
        # the strong-scaling reference point for the 8-GPU number
        from qpalm_b200 import batch as qb2
        bb = problems.mpc_batch(args.sweep_total, seed=args.seed)
        hh = qb2.Batch(bb.Q, bb.A, bb.settings, args.sweep_total)
        hh.upload(bb.q, bb.bmin, bb.bmax)
        hh.solve_resident(args.sweep_total)
        ms_sw = float(np.mean([hh.solve_resident(args.sweep_total) for _ in range(2)]))
        _, _, inf = hh.download(args.sweep_total)
        hh.cleanup()
        line["single_gpu_full_sweep"] = {"instances": args.sweep_total, "ms": ms_sw, "solves_per_sec": args.sweep_total / (ms_sw * 1e-3),
                                         "solved": sum(1 for i in inf if i["status_val"] == 1),
                                         "note": "all instances of the sweep on one GPU (multi-wave); 8-GPU strong-scaling efficiency = "
                                                 "(8-GPU solves/s) / (8 x this)"}
    if workload == "mpc_batch" and world > 1 and not args.no_dense:
        # BASELINE config 3 on N GPUs rides along: ONE dense QP, constraint rows sharded over the ranks (csrc/shard.cu, NCCL)
        from qpalm_b200 import rowshard
        rowshard.init(rank, world, torch.device("cuda", local))
        dense, p = bench_dense(args, lib, 1, 1, sample_clocks=False)
        t = torch.tensor([dense["ms_per_solve"], dense["e2e_s"]], device="cuda", dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        if rank == 0:
            line["time_to_solution"] = {"workload": f"dense random convex QP n={args.n} m={args.m} eps 1e-6, constraint rows sharded over {world} GPUs (NCCL)",
                                        "seconds": float(t[0]) * 1e-3, "e2e_seconds": float(t[1]), "status": dense["status"], "iter": dense["iter"],
                                        "iter_out": dense["iter_out"], "refactorizations": dense["refactorizations"],
                                        "updown_sweeps": dense["updown_sweeps"], "scaling": "strong"}
        rowshard.finalize()
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))


if __name__ == "__main__":
    main()
