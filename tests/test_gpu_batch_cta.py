"""The persistent batch engine's in-CTA linear algebra (batchp.cu) against float64 references, in both CTA shapes.

Shape 3 is the default build (32-column panels, 16-wide sub-panels, 3 CTAs per SM); shape 4 the -DQB_BP_VARIANT4 build
(24-column panels, 8-wide sub-panels, 4 CTAs per SM, a global-memory ping-pong buffer in the sort), which the solver picks
for 3 SMs < nb <= 4 SMs instances: the benchmark's 512 instances per GPU.  The probes (qpalm_b200_batchp_probe_*) run the
engine's own SYRK, Cholesky with the fused forward substitution, triangular solves, rank-k update sweeps and radix sort
on caller data, with the kernel's CTA size, shared-memory plan and persistent work queue.

Tolerances are a-priori rounding-error bounds with u = eps / 2 (Higham, Accuracy and Stability of Numerical Algorithms,
2nd ed.: gamma_k = k u / (1 - k u)), so a wrong entry fails and rounding does not.  The solver-level cases at the end choose
the engine and shape through nb, as a user does, and check them with last_shape."""
import ctypes as C

import numpy as np
import pytest

from qpalm_b200 import abi, problems
from qpalm_b200 import batch as qb
from qpalm_b200.interface import load_library
from test_gpu_batch import _check_instances, _rel

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
SHAPES = (3, 4)


@pytest.fixture(params=SHAPES, ids=["shape3", "shape4"])
def shape(request):
    return request.param


def _lib():
    lib = load_library("b200")
    if not getattr(lib, "_probe_typed", False):
        fp, ip, ci = abi.c_float_p, abi.c_int_p, abi.c_int
        lib.qpalm_b200_batchp_probe_newton.argtypes = [ci, ci, ci, ci, fp, fp, ci, C.c_double, ip, ip, fp, C.c_double, fp,
                                                       fp, fp, fp, fp, ip]
        lib.qpalm_b200_batchp_probe_newton.restype = C.c_int
        lib.qpalm_b200_batchp_probe_sort.argtypes = [ci, ci, ci, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
        lib.qpalm_b200_batchp_probe_sort.restype = C.c_int
        lib._probe_typed = True
    return lib


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def probe_newton(shape, A, insts, beta=0.0, from_q=None, sscale=1.0):
    """One probe call.  A: m x n (row c is column c of A').  insts: dicts with H0 (n x n symmetric; omitted with from_q),
    rhs, and optional pos / neg / upd = (rows, weights) and kpos.  Returns H, L (lower triangles), d_fused, d_after, info."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    m, n = A.shape
    nb = len(insts)
    cnt = np.zeros((nb, 4), np.int64)
    lists = np.zeros((nb, 3, m), np.int64)
    wts = np.zeros((nb, 3, m))
    for b, it in enumerate(insts):
        for s, key in enumerate(("pos", "neg", "upd")):
            rows, w = it.get(key, ((), ()))
            cnt[b, s] = len(rows)
            lists[b, s, :len(rows)] = rows
            wts[b, s, :len(rows)] = w
        cnt[b, 3] = it.get("kpos", 0)
    # column-major n x n on the C side: pass the transposes
    H0 = np.ascontiguousarray(from_q.T if from_q is not None else np.stack([it["H0"].T for it in insts]), dtype=np.float64)
    rhs = np.ascontiguousarray(np.stack([it["rhs"] for it in insts]), dtype=np.float64)
    H, L = np.zeros((nb, n, n)), np.zeros((nb, n, n))
    dfu, daf = np.zeros((nb, n)), np.zeros((nb, n))
    info = np.zeros(nb, np.int64)
    rc = _lib().qpalm_b200_batchp_probe_newton(shape, nb, n, m, abi.fptr(A), abi.fptr(H0), int(from_q is not None), sscale,
                                               abi.iptr(cnt), abi.iptr(lists), abi.fptr(wts), beta, abi.fptr(rhs), abi.fptr(H),
                                               abi.fptr(L), abi.fptr(dfu), abi.fptr(daf), abi.iptr(info))
    assert rc == 0, rc
    return H.transpose(0, 2, 1), L.transpose(0, 2, 1), dfu, daf, info


def probe_sort(shape, keys, vals):
    keys, vals = np.ascontiguousarray(keys, np.uint64).copy(), np.ascontiguousarray(vals, np.uint32).copy()
    nb, N = keys.shape
    rc = _lib().qpalm_b200_batchp_probe_sort(shape, nb, N, keys.ctypes.data_as(C.POINTER(C.c_uint64)),
                                             vals.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert rc == 0, rc
    return keys, vals


# ------------------------------------------------------------------------------------------------
# references and bounds
# ------------------------------------------------------------------------------------------------
def spd(rng, n, cond, scale=2.5):
    """Symmetric positive definite with eigenvalues scale * geomspace(1, 1 / cond)."""
    U, _ = np.linalg.qr(rng.standard_normal((n, n)))
    H = (U * (scale * np.geomspace(1.0, 1.0 / cond, n))) @ U.T
    return (H + H.T) / 2


def base(rng, n):
    """Well-conditioned SPD base of the update tests: eigenvalues in about [1, 5]."""
    M = rng.standard_normal((n, n)) / np.sqrt(n)
    return M @ M.T + np.eye(n)


def gram(A, rows, w):
    W = np.asarray(w)[:, None] * A[np.asarray(rows, dtype=np.int64)]
    return W.T @ W


def sym(Hl):
    return np.tril(Hl) + np.tril(Hl, -1).T


def check_factor(L, M, what):
    """Backward error of a Cholesky factor (Higham Thm 10.3): L L' = M + dM, |dM| <= gamma_{n+1} |L||L'| entrywise.  The
    bound is taken four times over: the blocked order of the kernel and the float64 rounding of L L' formed here (gamma_n
    |L||L'|) fit in it, a wrong entry of relative size 1e-12 does not."""
    n = len(L)
    assert np.all(np.diag(L) > 0), what
    LL = np.abs(L) @ np.abs(L).T
    err = np.abs(L @ L.T - M)
    tol = 4 * (n + 1) * EPS * LL
    assert np.all(err <= tol), (what, float(np.max(err / np.maximum(tol, 1e-300))))


def check_forward(L, Lref, M, what, extra=1.0):
    """Forward error against another factor of M: the backward error above (max entry <= 4 (n + 1) eps max|L||L'|) turns into
    a forward error of at most kappa(M) times it (Sun's perturbation bound for the Cholesky factor, with a factor n for
    the max norm against the Frobenius norm), relative to max|L|.  `extra` widens it where both factors carry rounding."""
    n = len(L)
    ev = np.linalg.eigvalsh(M)
    kappa = ev[-1] / ev[0]
    tol = extra * 4 * (n + 1) * n * EPS * kappa * np.max(np.abs(Lref))
    err = np.max(np.abs(L - Lref))
    assert err <= tol, (what, err, tol)


def check_solve(d, M, L, rhs, what, dM=0.0):
    """Backward error of (L L')^{-1} rhs (Higham Thm 10.4): (M + dM') d = rhs with |dM'| <= gamma_{3n+1} |L||L'|, four times
    over as above, plus the float64 rounding of the residual formed here (n eps (|M||d| + |rhs|)).  dM bounds |L L' - M|
    entrywise when L is not a factorisation of M itself (after update sweeps): it adds dM * sum|d| to every component."""
    n = len(L)
    ad = np.abs(d)
    r = np.abs(rhs - M @ d)
    tol = 4 * (3 * n + 1) * EPS * ((np.abs(L) @ (np.abs(L).T @ ad))) + n * EPS * (np.abs(M) @ ad + np.abs(rhs)) + dM * ad.sum()
    assert np.all(np.isfinite(d)), what
    assert np.all(r <= tol), (what, float(np.max(r / np.maximum(tol, 1e-300))))


def updated_bound(n, nup, S):
    """Entrywise bound on |L L' - H_final| after nup ranks of update sweeps.  The recurrence (chain warp and row owners) has
    no componentwise a-priori bound, so a normwise one: every rank passes each entry of the running factor through O(1)
    roundings per column, about (n + 1) u relative, and entries of L L' are bounded by S, the largest diagonal entry of any
    intermediate matrix.  The leaving rows are kept well inside the matrix (w' H^{-1} w about 1/2), so the downdates do not
    amplify it.  32 (n + nup) eps S is a margin of 16 over that; a lost rank or a wrong coefficient is off by O(S)."""
    return 32 * (n + nup) * EPS * S


# ------------------------------------------------------------------------------------------------
# SYRK lists
# ------------------------------------------------------------------------------------------------
SYRK_LENGTHS = (0, 1, 3, 4, 5, 7, 8, 9, 23, 24, 25, 31, 32, 33, 64, 100)


@pytest.mark.parametrize("n", [45, 240])
def test_syrk_lists(shape, n):
    """H = H0 + A_P' diag(w^2) A_P - A_N' diag(w^2) A_N for list lengths across both panel widths (24, 32) and the 4-column
    padding of the DMMA loop, weights over 1e-2 .. 1e3."""
    rng = np.random.default_rng(100 + n)
    m = 128
    A = rng.standard_normal((m, n))
    insts = []
    for i, K in enumerate(SYRK_LENGTHS):
        Kn = SYRK_LENGTHS[-1 - i]
        pr, nr = rng.choice(m, K, replace=False), rng.choice(m, Kn, replace=False)
        pw, nw = 10 ** rng.uniform(-2, 3, K), 10 ** rng.uniform(-2, 3, Kn)
        H0 = spd(rng, n, 10.0) + gram(A, nr, nw)    # the leaving rows are part of H0: H stays positive definite
        insts.append(dict(H0=H0, pos=(pr, pw), neg=(nr, nw), rhs=rng.standard_normal(n), T=(pr, pw, nr, nw)))
    H, L, dfu, daf, info = probe_newton(shape, A, insts)
    for b, it in enumerate(insts):
        pr, pw, nr, nw = it["T"]
        ref = it["H0"] + gram(A, pr, pw) - gram(A, nr, nw)
        # each entry is H0_ij plus K = |P| + |N| products of the rounded w a (two chunked DMMA sums and two final adds):
        # gamma_{K+3} T_ij, T = |H0| + sum w^2 |a_i a_j|; the float64 reference adds gamma_{K+1} T_ij; 2 (K + 4) eps covers both
        T = np.abs(it["H0"]) + gram(np.abs(A), pr, pw) + gram(np.abs(A), nr, nw)
        tol = 2 * (len(pr) + len(nr) + 4) * EPS * T
        err = np.abs(np.tril(H[b]) - np.tril(ref))
        assert np.all(err <= np.tril(tol)), (b, len(pr), len(nr), float(np.max(err - tol)))
        assert info[b] == 0
        check_factor(L[b], sym(H[b]), ("syrk factor", b))


# ------------------------------------------------------------------------------------------------
# factorisation and solves
# ------------------------------------------------------------------------------------------------
FACTOR_N = (1, 2, 7, 8, 9, 15, 16, 17, 23, 24, 25, 31, 32, 33, 47, 48, 49, 63, 64, 65, 95, 96, 97, 127, 128, 129,
            191, 192, 193, 239, 240)


@pytest.mark.parametrize("n", FACTOR_N)
def test_factor_and_solve(shape, n):
    """L = chol(H + beta I) and (L L')^{-1} rhs at every panel / sub-panel / 128-row boundary, condition numbers 1e1 and 1e8,
    beta in {0, 1e-7, 1}; then the f.fq path, which factors sscale * Q straight from the shared matrix (lds = n != ld)."""
    rng = np.random.default_rng(200 + n)
    A = rng.standard_normal((4, n))
    I = np.eye(n)
    for beta in (0.0, 1e-7, 1.0):
        insts = [dict(H0=spd(rng, n, cond), rhs=rng.standard_normal(n)) for cond in (1e1, 1e8)]
        H, L, dfu, daf, info = probe_newton(shape, A, insts, beta=beta)
        for b, it in enumerate(insts):
            what = (n, beta, b)
            M = it["H0"] + beta * I
            assert info[b] == 0, what
            assert np.array_equal(H[b], np.tril(it["H0"])), what
            check_factor(L[b], M, what)
            check_forward(L[b], np.linalg.cholesky(M), M, what, extra=2.0)
            check_solve(dfu[b], M, L[b], it["rhs"], what)
            # no update: the fused forward substitution and the separate one read the same panel values and 1 / l_jj
            assert np.array_equal(dfu[b], daf[b]), what
    Q, sscale, beta = spd(rng, n, 1e1), 0.37, 1e-7
    insts = [dict(rhs=rng.standard_normal(n)) for _ in range(3)]
    H, L, dfu, daf, info = probe_newton(shape, A, insts, beta=beta, from_q=Q, sscale=sscale)
    M = sscale * Q + beta * I
    for b, it in enumerate(insts):
        what = ("from_q", n, b)
        assert info[b] == 0, what
        assert np.array_equal(H[b], np.tril(sscale * Q)), what
        check_factor(L[b], M, what)
        check_solve(dfu[b], M, L[b], it["rhs"], what)
        assert np.array_equal(dfu[b], daf[b]), what
        assert np.array_equal(L[b], L[0]), what


# ------------------------------------------------------------------------------------------------
# rank-k update sweeps
# ------------------------------------------------------------------------------------------------
UPD_N = (1, 5, 16, 17, 31, 32, 33, 48, 63, 64, 65, 200, 239, 240)
UPD_K = (1, 7, 8, 9, 16, 17, 40)    # 40: the engine's default cap on the ranks of one update


def _update_case(rng, A, B, k, kpos):
    m = A.shape[0]
    rows, w = rng.choice(m, k, replace=False), rng.uniform(0.5, 1.5, k)
    H0 = B + gram(A, rows[kpos:], w[kpos:])      # the leaving rows are part of H0, as in QPALM
    Hf = B + gram(A, rows[:kpos], w[:kpos])
    S = np.max(np.diag(H0 + gram(A, rows[:kpos], w[:kpos])))
    rhs = rng.standard_normal(A.shape[1])
    sweep = dict(H0=H0, upd=(rows, w), kpos=kpos, rhs=rhs)
    refac = dict(H0=H0, pos=(rows[:kpos], w[:kpos]), neg=(rows[kpos:], w[kpos:]), rhs=rhs)
    return sweep, refac, Hf, S


@pytest.mark.parametrize("n", UPD_N)
def test_update_sweeps(shape, n):
    """Rank-k update of L in sweeps of 8 ranks, entering rows first: k across one / several sweeps, kpos = 0, k, 3 (both
    signs inside one sweep) and k - 1.  The final L against numpy's factor of the modified matrix and against the probe's
    own refactorisation (the same rows through the SYRK lists); (L L')^{-1} rhs with the updated L and rdiag; and update
    followed by downdate of the same rows against the original factor."""
    rng = np.random.default_rng(300 + n)
    m = 96
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    B = base(rng, n)
    insts, cases = [dict(H0=B, rhs=rng.standard_normal(n))], []
    for k in UPD_K:
        for kpos in sorted({0, k, min(3, k), k - 1}):
            sweep, refac, Hf, S = _update_case(rng, A, B, k, kpos)
            cases.append(("sweep", len(insts), len(insts) + 1, k, kpos, Hf, S))
            insts += [sweep, refac]
        rows, w = rng.choice(m, k, replace=False), rng.uniform(0.5, 1.5, k)
        cases.append(("round trip", len(insts), 0, k, k, B, np.max(np.diag(B + gram(A, rows, w)))))
        insts.append(dict(H0=B, upd=(np.concatenate([rows, rows]), np.concatenate([w, w])), kpos=k, rhs=rng.standard_normal(n)))
    H, L, dfu, daf, info = probe_newton(shape, A, insts)
    assert not np.any(info), info
    check_factor(L[0], B, "base")
    for kind, b, ref, k, kpos, Hf, S in cases:
        what = (kind, n, k, kpos)
        nup = len(insts[b]["upd"][0])
        check_solve(dfu[b], insts[b]["H0"], L[b], insts[b]["rhs"], what + ("fused",))
        assert np.all(np.diag(L[b]) > 0), what
        dM = updated_bound(n, nup, S)
        err = np.max(np.abs(L[b] @ L[b].T - Hf))
        assert err <= dM, (what, err, dM)
        check_forward(L[b], np.linalg.cholesky(Hf), Hf, what + ("numpy",), extra=8.0)
        check_forward(L[b], L[ref], Hf, what + ("probe",), extra=8.0)   # the refactorisation, or the original factor
        check_solve(daf[b], Hf, L[b], insts[b]["rhs"], what + ("after",), dM=dM)


# ------------------------------------------------------------------------------------------------
# many instances per launch, failing downdates
# ------------------------------------------------------------------------------------------------
def _grid(shape):
    return shape * _sms()     # shared memory admits exactly `shape` CTAs per SM


def test_failing_downdates_among_healthy_instances(shape):
    """nb = 2 grid + 3 instances, each with its own matrix, so every CTA runs several: every third downdates a row that
    H0 does not contain (w' H0^{-1} w > 1: definiteness is lost, info bit 0), the others take a healthy mixed sweep and must
    still be exact.  The chain warp keeps walking every column and arriving on every barrier after a non-positive pivot
    (ud_chain_role only records it), so the mbarrier phases stay in step for the CTA's next instance."""
    n, m = 37, 24
    nb = 2 * _grid(shape) + 3
    rng = np.random.default_rng(400 + shape)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    insts, refs = [], []
    for b in range(nb):
        B = base(rng, n)
        if b % 3 == 1:
            rows, w = rng.choice(m, 2, replace=False), np.array([4.0, 4.0])
            v = w[0] * A[rows[0]]
            assert v @ np.linalg.solve(B, v) > 1.0
            insts.append(dict(H0=B, upd=(rows, w), kpos=0, rhs=rng.standard_normal(n)))
            refs.append(None)
        else:
            sweep, _, Hf, S = _update_case(rng, A, B, 9, 4)
            insts.append(sweep)
            refs.append((Hf, S))
    H, L, dfu, daf, info = probe_newton(shape, A, insts)
    for b, ref in enumerate(refs):
        if ref is None:
            assert info[b] == 1, (b, info[b])
            continue
        Hf, S = ref
        assert info[b] == 0, (b, info[b])
        dM = updated_bound(n, 9, S)
        assert np.max(np.abs(L[b] @ L[b].T - Hf)) <= dM, b
        check_solve(daf[b], Hf, L[b], insts[b]["rhs"], ("healthy", b), dM=dM)


def test_identical_instances_give_identical_results(shape):
    """nb = 2 grid + 3 copies of one instance (SYRK lists, factorisation, a two-sweep mixed update): per-instance strides and
    offsets, and the mbarrier phase a CTA carries from one instance to the next, must not change a single bit."""
    n, m = 53, 40
    nb = 2 * _grid(shape) + 3
    rng = np.random.default_rng(500 + shape)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    B = base(rng, n)
    sweep, _, Hf, S = _update_case(rng, A, B, 13, 5)
    pr, nr = rng.choice(m, 6, replace=False), rng.choice(m, 3, replace=False)
    pw, nw = rng.uniform(0.5, 1.5, 6), rng.uniform(0.5, 1.5, 3)
    H0 = sweep["H0"] + gram(A, nr, nw)
    inst = dict(sweep, H0=H0, pos=(pr, pw), neg=(nr, nw))
    H, L, dfu, daf, info = probe_newton(shape, A, [inst] * nb)
    assert not np.any(info)
    for X in (H, L, dfu, daf):
        assert all(np.array_equal(X[b], X[0]) for b in range(1, nb))
    Hn = sym(H[0])    # the SYRK result the factorisation started from (checked against its reference in test_syrk_lists)
    assert np.max(np.abs(Hn - (H0 + gram(A, pr, pw) - gram(A, nr, nw)))) <= 2 * (9 + 4) * EPS * np.max(np.abs(Hn)) * n
    check_solve(dfu[0], Hn, np.linalg.cholesky(Hn), inst["rhs"], "fused")
    Hfin = Hf + gram(A, pr, pw)      # + the entering rows - the leaving rows of the sweeps
    dM = updated_bound(n, 13, S + np.max(np.diag(gram(A, pr, pw))))
    assert np.max(np.abs(L[0] @ L[0].T - Hfin)) <= dM
    check_solve(daf[0], Hfin, L[0], inst["rhs"], "after", dM=dM)


# ------------------------------------------------------------------------------------------------
# sort
# ------------------------------------------------------------------------------------------------
SORT_N = (1, 2, 3, 31, 32, 33, 255, 256, 257, 1000, 2047, 2048)
KEYSETS = ("breakpoints", "all_equal", "low_byte", "high_byte", "duplicates")


def _keys(rng, kind, N):
    full = lambda size: rng.integers(0, 2 ** 64, size, dtype=np.uint64)   # noqa: E731
    if kind == "breakpoints":    # the line search's keys: bit patterns of positive doubles, +inf, and ~0 for s <= 0
        k = np.exp(rng.uniform(-30, 30, N)).view(np.uint64).copy()
        sel = rng.random(N)
        k[sel < 0.1] = np.uint64(0x7FF0000000000000)
        k[(sel >= 0.1) & (sel < 0.3)] = np.uint64(0xFFFFFFFFFFFFFFFF)
        return k
    if kind == "all_equal":      # every digit constant: no pass runs
        return np.full(N, full(1)[0], dtype=np.uint64)
    if kind == "low_byte":       # one pass (digit 0)
        return (full(1)[0] & np.uint64(~0xFF & 0xFFFFFFFFFFFFFFFF)) | rng.integers(0, 256, N, dtype=np.uint64)
    if kind == "high_byte":      # one pass (digit 7)
        return (full(1)[0] & np.uint64(0x00FFFFFFFFFFFFFF)) | (rng.integers(0, 256, N, dtype=np.uint64) << np.uint64(56))
    return rng.choice(full(3), N)   # heavy duplication, eight passes


@pytest.mark.parametrize("kind", KEYSETS)
def test_sort(shape, kind):
    """p_sort against a stable argsort.  The passes over constant digits are skipped, so these key sets perform 0, 1 and
    8 passes: the final copy back (kin != kg) is taken and skipped in both builds (in shape 4 the ping-pong buffer is the
    global array itself)."""
    rng = np.random.default_rng(600 + KEYSETS.index(kind))
    for N in SORT_N:
        keys = np.stack([_keys(rng, kind, N) for _ in range(3)])
        vals = np.tile(np.arange(N, dtype=np.uint32), (3, 1))
        ks, vs = probe_sort(shape, keys, vals)
        for b in range(3):
            order = np.argsort(keys[b], kind="stable")
            assert np.array_equal(ks[b], keys[b][order]), (kind, N, b)
            assert np.array_equal(vs[b], vals[b][order]), (kind, N, b)


# ------------------------------------------------------------------------------------------------
# solver level: the shape the engine selects
# ------------------------------------------------------------------------------------------------
def _solve(b, lo=0, hi=None):
    hi = b.q.shape[0] if hi is None else hi
    h = qb.Batch(b.Q, b.A, b.settings, hi - lo)
    assert h.ok
    xs, ys, infos = h.solve(b.q[lo:hi], b.bmin[lo:hi], b.bmax[lo:hi])
    shape = h.last_shape()
    h.cleanup()
    return xs, ys, infos, shape


def test_shape4_small_instances_against_oracle():
    """3 SMs + 1 instances select the 4-CTAs-per-SM build; every instance against the oracle."""
    nb = 3 * _sms() + 1
    b = problems.mpc_batch(nb, n=48, m0=80, seed=31)
    xs, ys, infos, shape = _solve(b)
    assert shape == 4
    _check_instances(b, range(nb), xs, ys, infos)


def test_shape4_benchmark_size_against_shape3():
    """The benchmark's instance size (n = 240, m = 949) in the build the benchmark runs (shape 4, 3 SMs + 1 instances),
    every instance against the same instances solved by the default build (batches of 3 SMs and 1), eight sampled ones,
    the one with the most iterations among them, against the oracle."""
    nb = 3 * _sms() + 1
    b = problems.mpc_batch(nb, seed=2)
    x4, y4, i4, s4 = _solve(b)
    assert s4 == 4
    x3a, y3a, i3a, s3a = _solve(b, 0, nb - 1)
    x3b, y3b, i3b, s3b = _solve(b, nb - 1, nb)
    assert s3a == 3 and s3b == 3
    x3, y3, i3 = np.vstack([x3a, x3b]), np.vstack([y3a, y3b]), i3a + i3b
    for k in range(nb):
        g, r = i4[k], i3[k]
        assert g["status_val"] == r["status_val"], (k, g, r)
        assert abs(g["iter"] - r["iter"]) <= max(1, int(np.ceil(0.05 * r["iter"]))), (k, g["iter"], r["iter"])
        assert abs(g["iter_out"] - r["iter_out"]) <= 1, (k, g["iter_out"], r["iter_out"])
        if r["status_val"] == 1:
            assert _rel(x4[k], x3[k]) < 1e-7 and _rel(y4[k], y3[k]) < 1e-7, k
            assert abs(g["objective"] - r["objective"]) <= 1e-7 * max(1.0, abs(r["objective"]))
    worst = int(np.argmax([i["iter"] for i in i4]))
    sample = sorted({0, 1, nb // 3, nb // 2, 2 * nb // 3, nb - 2, nb - 1, worst})
    _check_instances(b, sample, x4, y4, i4)


@pytest.mark.parametrize("n,m0,window,expected", [
    (240, 720, True, 4),     # m = 960: the largest m of the shape-4 build (VS_LEN)
    (240, 721, True, 3),     # m = 961: shape 4 refuses, the default build takes the batch
    (240, 784, False, 3),    # m = 1024: 2m = 2048, the largest in-CTA sort
    (240, 785, False, 0),    # m = 1025: the lock-step engine
    (241, 100, False, 0),    # n = 241: beyond NMAX, the lock-step engine
], ids=["m960_shape4", "m961_shape3", "m1024_shape3", "m1025_lockstep", "n241_lockstep"])
def test_engine_and_shape_limits(n, m0, window, expected):
    nb = 3 * _sms() + 1 if window else 3
    b = problems.mpc_batch(nb, n=n, m0=m0, seed=41)
    xs, ys, infos, shape = _solve(b)
    assert shape == expected
    _check_instances(b, sorted({0, nb // 2, nb - 1}), xs, ys, infos)
