"""Host-side mirror of the sparse Newton-system operator ABI (include/qpalm_b200.h, csrc/sparse*.cu).

`symbolic(Q, A)` runs the library's one-time symbolic analysis (no CUDA call) and returns its arrays; `sparse_newton(...)`
drives factor + rank update/downdate + solve on the GPU.  Replaces cholmod_analyze / cholmod_factorize / cholmod_updown /
cholmod_solve as used by /root/reference/src/solver_interface.c:319-519 for problems with a sparse Schur complement.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import abi
from .interface import load_library

_ARRAYS = ("perm", "iperm", "sn_first", "sn_of_col", "rows_off", "rowidx", "rel", "sn_parent", "child_ptr", "child_idx",
           "lvl_ptr", "lvl_sn", "panel_off", "upd_off")


def _lib():
    lib = load_library("b200")
    lib.qpalm_b200_symbolic_analyze.restype = C.c_void_p
    lib.qpalm_b200_symbolic_analyze.argtypes = [C.POINTER(abi.SolverSparse), C.POINTER(abi.SolverSparse)]
    lib.qpalm_b200_symbolic_info.argtypes = [C.c_void_p, abi.c_int_p, C.POINTER(C.c_double)]
    lib.qpalm_b200_symbolic_array.restype = abi.c_int
    lib.qpalm_b200_symbolic_array.argtypes = [C.c_void_p, C.c_char_p, abi.c_int_p, abi.c_int]
    lib.qpalm_b200_symbolic_free.argtypes = [C.c_void_p]
    lib.qpalm_b200_sparse_newton.argtypes = [C.POINTER(abi.SolverSparse), C.POINTER(abi.SolverSparse), abi.c_float_p, abi.c_int_p,
                                             C.c_double, abi.c_float_p, abi.c_float_p, abi.c_float_p, abi.c_int_p, abi.c_int_p,
                                             abi.c_int, abi.c_int_p, abi.c_int, abi.c_float_p]
    lib.qpalm_b200_sparse_ldl.argtypes = [C.POINTER(abi.SolverSparse), abi.c_int, abi.c_float_p, abi.c_float_p, abi.c_float_p,
                                          abi.c_int_p, abi.c_float_p, abi.c_int, abi.c_int_p]
    lib.qpalm_b200_kkt_newton.argtypes = [C.POINTER(abi.SolverSparse), C.POINTER(abi.SolverSparse), abi.c_float_p, abi.c_int_p,
                                          C.c_double, abi.c_float_p, abi.c_float_p, abi.c_int_p, abi.c_float_p]
    return lib


def symbolic(Q: abi.CSC, A: abi.CSC | None) -> dict:
    lib = _lib()
    h = lib.qpalm_b200_symbolic_analyze(Q.ptr(), A.ptr() if A is not None else None)
    if not h:
        raise RuntimeError("symbolic analysis failed")
    try:
        info = np.zeros(8, dtype=np.int64)
        flops = C.c_double(0)
        lib.qpalm_b200_symbolic_info(h, abi.iptr(info), C.byref(flops))
        out = dict(zip(("n", "nsuper", "nlevels", "max_ns", "max_nf", "nnzS", "nnzL", "upd_entries"), (int(v) for v in info)))
        out["flops"] = flops.value
        for name in _ARRAYS:
            ln = int(lib.qpalm_b200_symbolic_array(h, name.encode(), None, 0))
            a = np.zeros(max(ln, 1), dtype=np.int64)
            lib.qpalm_b200_symbolic_array(h, name.encode(), abi.iptr(a), ln)
            out[name] = a[:ln]
        return out
    finally:
        lib.qpalm_b200_symbolic_free(h)


def sparse_newton(Q: abi.CSC, A: abi.CSC | None, sigma, active, beta, rhs, enter=(), leave=(), want_factor=False, want_bound=False):
    """d = (Q + A_J' Sigma_J A_J (+ enter, - leave) + beta I)^{-1} rhs through the supernodal factor.
    Returns (d, L_permuted or None, perm or None, gershgorin bound or None)."""
    lib = _lib()
    n = Q.ncol
    m = A.nrow if A is not None else 0
    sigma = np.ascontiguousarray(sigma if m else np.zeros(1), dtype=np.float64)
    act = np.ascontiguousarray(active if m else np.zeros(1), dtype=np.int64)
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    d = np.zeros(n)
    L = np.zeros((n, n), order="F") if want_factor else None
    perm = np.zeros(n, dtype=np.int64) if want_factor else None
    en = np.ascontiguousarray(enter if len(enter) else [0], dtype=np.int64)
    lv = np.ascontiguousarray(leave if len(leave) else [0], dtype=np.int64)
    bound = np.zeros(1) if want_bound else None
    rc = lib.qpalm_b200_sparse_newton(Q.ptr(), A.ptr() if A is not None else None, abi.fptr(sigma), abi.iptr(act), float(beta),
                                      abi.fptr(rhs), abi.fptr(d),
                                      L.ctypes.data_as(abi.c_float_p) if want_factor else None,
                                      abi.iptr(perm) if want_factor else None, abi.iptr(en), len(enter), abi.iptr(lv), len(leave),
                                      abi.fptr(bound) if want_bound else None)
    if rc:
        raise RuntimeError(f"qpalm_b200_sparse_newton failed with code {rc}")
    return d, L, perm, (float(bound[0]) if want_bound else None)


def sparse_ldl(K: abi.CSC, n_pos: int, rhs, want_factor=False, panels_len=0):
    """x = K^{-1} rhs through the signed supernodal factorization K(perm, perm) = L S L' of a quasi-definite K (lower
    triangle CSC; original columns >= n_pos carry negative pivots), one solve without refinement.
    Returns (rc, x, L_permuted or None, perm or None, panels or None): rc is 0, or 1000 + info when a pivot did not
    have its a-priori sign (info - 1: a permuted column in the front of such a pivot or
    in a front above it).  panels_len > 0 (symbolic(K, None)["nnzL"]) also returns the raw factor panels."""
    lib = _lib()
    N = K.ncol
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    x = np.zeros(N)
    L = np.zeros((N, N), order="F") if want_factor else None
    perm = np.zeros(N, dtype=np.int64) if want_factor else None
    panels = np.zeros(max(panels_len, 1)) if panels_len else None
    plen = np.zeros(1, dtype=np.int64)
    rc = lib.qpalm_b200_sparse_ldl(K.ptr(), int(n_pos), abi.fptr(rhs), abi.fptr(x),
                                   L.ctypes.data_as(abi.c_float_p) if want_factor else None,
                                   abi.iptr(perm) if want_factor else None,
                                   abi.fptr(panels) if panels_len else None, int(panels_len), abi.iptr(plen))
    if rc and rc < 1000:
        raise RuntimeError(f"qpalm_b200_sparse_ldl failed with code {rc}")
    if panels_len:
        assert int(plen[0]) == panels_len, (int(plen[0]), panels_len)
    return rc, x, L, perm, panels


def kkt_newton(Q: abi.CSC, A: abi.CSC, sigma, active, beta, rhs):
    """The KKT Newton step: d = (Q + A_J' Sigma_J A_J + beta I)^{-1} rhs through the L S L' factorization of
    [Q + beta I, A_J'; A_J, -inv(Sigma_J)] and the solver's iterative refinement.
    Returns (rc, d, refinement corrections applied, (|res|inf, ref) of the last residual)."""
    lib = _lib()
    sigma = np.ascontiguousarray(sigma, dtype=np.float64)
    act = np.ascontiguousarray(active, dtype=np.int64)
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    d = np.zeros(Q.ncol)
    refine = np.zeros(1, dtype=np.int64)
    norms = np.zeros(2)
    rc = lib.qpalm_b200_kkt_newton(Q.ptr(), A.ptr(), abi.fptr(sigma), abi.iptr(act), float(beta), abi.fptr(rhs), abi.fptr(d),
                                   abi.iptr(refine), abi.fptr(norms))
    if rc and rc < 1000:
        raise RuntimeError(f"qpalm_b200_kkt_newton failed with code {rc}")
    return rc, d, int(refine[0]), (float(norms[0]), float(norms[1]))
