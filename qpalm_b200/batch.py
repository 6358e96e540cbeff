"""Python binding of the additive batch entry point (include/qpalm_b200.h Part 3)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import abi
from .abi import QPALMData, QPALMInfo, QPALMSettings, c_float_p, fptr
from .interface import load_library


def _lib():
    lib = load_library("b200")
    if not getattr(lib, "_batch_typed", False):
        lib.qpalm_b200_batch_setup.argtypes = [C.POINTER(QPALMData), C.POINTER(QPALMSettings), abi.c_int]
        lib.qpalm_b200_batch_setup.restype = C.c_void_p
        lib.qpalm_b200_batch_solve.argtypes = [C.c_void_p, abi.c_int, c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                               C.POINTER(QPALMInfo)]
        lib.qpalm_b200_batch_solve.restype = C.c_int
        lib.qpalm_b200_batch_upload.argtypes = [C.c_void_p, abi.c_int, c_float_p, c_float_p, c_float_p]
        lib.qpalm_b200_batch_upload.restype = C.c_int
        lib.qpalm_b200_batch_solve_resident.argtypes = [C.c_void_p, abi.c_int, C.POINTER(C.c_double)]
        lib.qpalm_b200_batch_solve_resident.restype = C.c_int
        lib.qpalm_b200_batch_download.argtypes = [C.c_void_p, abi.c_int, c_float_p, c_float_p, C.POINTER(QPALMInfo)]
        lib.qpalm_b200_batch_download.restype = C.c_int
        lib.qpalm_b200_batch_warm_start.argtypes = [C.c_void_p, abi.c_int, c_float_p, c_float_p]
        lib.qpalm_b200_batch_warm_start.restype = C.c_int
        lib.qpalm_b200_batch_last_launches.argtypes = [C.c_void_p]
        lib.qpalm_b200_batch_last_launches.restype = C.c_longlong
        lib.qpalm_b200_batch_last_shape.argtypes = [C.c_void_p]
        lib.qpalm_b200_batch_last_shape.restype = C.c_int
        lib.qpalm_b200_batch_stats.argtypes = [C.c_void_p, abi.c_int, c_float_p]
        lib.qpalm_b200_batch_stats.restype = C.c_int
        lib.qpalm_b200_batch_syrk_stats.argtypes = [C.c_void_p, abi.c_int, c_float_p]
        lib.qpalm_b200_batch_syrk_stats.restype = C.c_int
        lib.qpalm_b200_batch_linesearch_stats.argtypes = [C.c_void_p, abi.c_int, c_float_p]
        lib.qpalm_b200_batch_linesearch_stats.restype = C.c_int
        lib.qpalm_b200_batch_cleanup.argtypes = [C.c_void_p]
        lib.qpalm_b200_batch_cleanup.restype = None
        lib._batch_typed = True
    return lib


class Batch:
    """nb QPs sharing (Q, A, settings); q, bmin, bmax per instance (rows)."""

    def __init__(self, Q, A, settings: dict, nb_max: int):
        self.lib = _lib()
        self.Q, self.A = Q, A
        self.n, self.m = Q.ncol, A.nrow
        st = QPALMSettings()
        self.lib.qpalm_set_default_settings.argtypes = [C.POINTER(QPALMSettings)]
        self.lib.qpalm_set_default_settings(C.byref(st))
        for k, v in settings.items():
            setattr(st, k, v)
        self.settings = st
        z = np.zeros(max(self.n, self.m, 1))
        d = QPALMData()
        d.n, d.m, d.Q, d.A = self.n, self.m, Q.ptr(), A.ptr()
        d.q, d.c, d.bmin, d.bmax = fptr(z), 0.0, fptr(z), fptr(z)
        self._keep = (z, d)
        self.h = self.lib.qpalm_b200_batch_setup(C.byref(d), C.byref(st), nb_max)
        self.nb_max = nb_max

    @property
    def ok(self):
        return bool(self.h)

    def warm_start(self, x=None, y=None):
        """Warm start of the next solve (qpalm_warm_start per instance): x is nb' x n, y is nb' x m, unscaled, as a solve
        returns them; instances k < nb' start from row k, the others cold.  Either may be None: that part starts cold.
        warm_start() with neither clears a pending warm start."""
        x = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        y = None if y is None else np.ascontiguousarray(y, dtype=np.float64)
        rows = None
        for name, a, cols in (("x", x, self.n), ("y", y, self.m)):
            if a is None:
                continue
            if a.ndim != 2 or a.shape[1] != cols:
                raise ValueError(f"warm start {name}: expected nb x {cols}, got shape {a.shape}")
            if rows is not None and a.shape[0] != rows:
                raise ValueError(f"warm start x and y have different row counts ({rows} and {a.shape[0]})")
            rows = a.shape[0]
        if rows is not None and not 1 <= rows <= self.nb_max:
            raise ValueError(f"warm start of {rows} instances: expected 1 to nb_max = {self.nb_max}")
        rc = self.lib.qpalm_b200_batch_warm_start(self.h, rows or 0, None if x is None else fptr(x), None if y is None else fptr(y))
        if rc:
            raise RuntimeError(f"qpalm_b200_batch_warm_start failed: {rc}")

    def solve(self, q, bmin, bmax, x=None, y=None, info=None, raw_info=False, x_ws=None, y_ws=None):
        """One call of the batch entry point with HOST buffers (H2D of q / bmin / bmax, solve, D2H of x / y / info).
        x, y, info: optional caller-owned result buffers (e.g. pinned memory) reused across calls; raw_info=True returns the
        QPALMInfo array itself instead of a list of dicts.  x_ws, y_ws: warm start of this solve (see warm_start)."""
        if x_ws is not None or y_ws is not None:
            self.warm_start(x_ws, y_ws)
        nb = q.shape[0]
        q, bmin, bmax = (np.ascontiguousarray(a, dtype=np.float64) for a in (q, bmin, bmax))
        if x is None:
            x = np.zeros((nb, self.n))
        if y is None:
            y = np.zeros((nb, self.m))
        if info is None:
            info = (QPALMInfo * nb)()
        rc = self.lib.qpalm_b200_batch_solve(self.h, nb, fptr(q), fptr(bmin), fptr(bmax), fptr(x), fptr(y), info)
        if rc:
            raise RuntimeError(f"qpalm_b200_batch_solve failed: {rc}")
        return x, y, (info if raw_info else _infos(info, nb))

    def upload(self, q, bmin, bmax):
        self._res = tuple(np.ascontiguousarray(a, dtype=np.float64) for a in (q, bmin, bmax))
        rc = self.lib.qpalm_b200_batch_upload(self.h, self._res[0].shape[0], *[fptr(a) for a in self._res])
        if rc:
            raise RuntimeError(f"batch_upload failed: {rc}")

    def solve_resident(self, nb):
        ms = C.c_double(0)
        rc = self.lib.qpalm_b200_batch_solve_resident(self.h, nb, C.byref(ms))
        if rc:
            raise RuntimeError(f"batch_solve_resident failed: {rc}")
        return ms.value

    def download(self, nb):
        x, y = np.zeros((nb, self.n)), np.zeros((nb, self.m))
        info = (QPALMInfo * nb)()
        rc = self.lib.qpalm_b200_batch_download(self.h, nb, fptr(x), fptr(y), info)
        if rc:
            raise RuntimeError(f"batch_download failed: {rc}")
        return x, y, _infos(info, nb)

    def stats(self, nb):
        out = np.zeros(8)
        if self.lib.qpalm_b200_batch_stats(self.h, nb, fptr(out)):
            raise RuntimeError("batch_stats failed")
        syrk = np.zeros(2)
        if self.lib.qpalm_b200_batch_syrk_stats(self.h, nb, fptr(syrk)):
            raise RuntimeError("batch_syrk_stats failed")
        ls = np.zeros(2)
        if self.lib.qpalm_b200_batch_linesearch_stats(self.h, nb, fptr(ls)):
            raise RuntimeError("batch_linesearch_stats failed")
        return dict(inner=out[0], outer=out[1], refactorizations=out[2], refactor_J_sum=out[3],
                    engine={1: "lockstep", 2: "persistent"}.get(int(out[4]), "?"),
                    updown_sweeps=out[5], updown_rank_sum=out[6], updown_failed=out[7],
                    syrk_entries=syrk[0], scratch_rebuilds=syrk[1], ls_breakpoints=ls[0], ls_walked=ls[1])

    def last_launches(self):
        return int(self.lib.qpalm_b200_batch_last_launches(self.h))

    def last_shape(self):
        """Engine of the last solve: 0 lock-step, 3 or 4 persistent with 3 or 4 CTAs per SM."""
        return int(self.lib.qpalm_b200_batch_last_shape(self.h))

    def cleanup(self):
        if self.h:
            self.lib.qpalm_b200_batch_cleanup(self.h)
            self.h = None


def _infos(info, nb):
    return [dict(status_val=int(info[k].status_val), iter=int(info[k].iter), iter_out=int(info[k].iter_out),
                 pri_res_norm=float(info[k].pri_res_norm), dua_res_norm=float(info[k].dua_res_norm),
                 objective=float(info[k].objective)) for k in range(nb)]


def available() -> bool:
    """True when the batch kernels are built into the library (probe with a 1-instance setup)."""
    try:
        from . import problems
        b = problems.mpc_batch(1, n=8, m0=4, seed=0)
        h = Batch(b.Q, b.A, b.settings, 1)
        ok = h.ok
        h.cleanup()
        return ok
    except Exception:
        return False


def solve_batch(b, nb_max=None, x_ws=None, y_ws=None):
    h = Batch(b.Q, b.A, b.settings, nb_max or b.q.shape[0])
    if not h.ok:
        raise RuntimeError("batch setup failed")
    try:
        return h.solve(b.q, b.bmin, b.bmax, x_ws=x_ws, y_ws=y_ws)
    finally:
        h.cleanup()
