"""The dense Newton system's kernels (dense.cu) against float64 references: the TMA-fed DMMA GEMM (both tile kernels), the
two-level blocked Cholesky (with and without the look-ahead schedule, single-matrix and batched with masks), the inverse-only
path of the diagonal-block kernel, and the triangular solves (the one-launch dataflow solve and the per-block launches).

The probes (qpalm_b200_dense_probe_*) call the production functions unchanged on caller data, on a fresh non-blocking stream.
Tolerances are a-priori rounding-error bounds with u = eps / 2 and gamma_k = k u / (1 - k u) (Higham, Accuracy and Stability
of Numerical Algorithms, 2nd ed.).  The Cholesky's panels and the solves multiply by explicitly inverted diagonal blocks, so
Higham's bounds for substitution (Thm 10.3, 8.5) do not hold as such: the bounds below add the triangular-inversion residual
terms (ch. 13-14), derived in the docstrings of check_inverse, check_factor and check_solve.  The negative controls at the
end (no GPU needed) show that each check rejects a result one entry of which is off by a relative 1e-12, and a GEMM result
missing one k-tile."""
import ctypes as C

import numpy as np
import pytest

from qpalm_b200 import abi, problems
from qpalm_b200 import batch as qb
from qpalm_b200.interface import load_library
from test_gpu_batch import _check_instances
from test_gpu_batch_cta import EPS, base, spd


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def gpu(f):
    """The GPU cases: marked `gpu` and skipped without a device, so that the host-only negative controls run anywhere."""
    return pytest.mark.gpu(pytest.mark.skipif(not _has_gpu(), reason="no CUDA device")(f))


U = EPS / 2
NB = 128


def gamma(k):
    return k * U / (1 - k * U)


# ------------------------------------------------------------------------------------------------
# probes
# ------------------------------------------------------------------------------------------------
def _lib():
    lib = load_library("b200")
    if not getattr(lib, "_dense_probe_typed", False):
        fp, ip, ci, d = abi.c_float_p, abi.c_int_p, abi.c_int, C.c_double
        lib.qpalm_b200_dense_probe_gemm.argtypes = [ci, ci, ci, ci, ip, ip, fp, ci, ci, fp, ci, ci, fp, ci, ci, d, d, ci, ci, ip]
        lib.qpalm_b200_dense_probe_potrf.argtypes = [ci, ci, fp, fp, ip, ip, ci]
        lib.qpalm_b200_dense_probe_trtri.argtypes = [ci, fp, fp]
        lib.qpalm_b200_dense_probe_solve.argtypes = [ci, ci, fp, fp, fp, ci, ip, ip, ci, ip]
        for f in ("gemm", "potrf", "trtri", "solve"):
            getattr(lib, "qpalm_b200_dense_probe_" + f).restype = C.c_int
        lib._dense_probe_typed = True
    return lib


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _ints(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int64)


def _iptr(a):
    return None if a is None else abi.iptr(a)


def _colmajor(X):
    """Stack of matrices (nb, r, c) -> the column-major buffer (nb, c, r) C-contiguous."""
    return np.ascontiguousarray(np.swapaxes(X, -1, -2), dtype=np.float64)


def probe_gemm(A, B, C0, alpha, beta, Kz=None, mask=None, lower_only=False, in_place=False):
    """C = beta C0 + alpha A[:, :Kz] B[:, :Kz]' per instance.  A (nb, M, K), B (nb, N, K), C0 (nb, M, N); with in_place A is
    C0 itself (N = 128, K <= 128).  Returns (C, tile rows of the kernel that ran)."""
    nb, M, N = C0.shape
    K = B.shape[2]
    Ab = _colmajor(A if not in_place else np.zeros((1, 2, 2)))
    Bb, Cb = _colmajor(B), _colmajor(C0)
    kz, mk, rows = _ints(Kz), _ints(mask), np.zeros(1, np.int64)
    rc = _lib().qpalm_b200_dense_probe_gemm(nb, M, N, K, _iptr(kz), _iptr(mk), abi.fptr(Ab), M, M * K, abi.fptr(Bb), N, N * K,
                                            abi.fptr(Cb), M, M * N, float(alpha), float(beta), int(lower_only), int(in_place),
                                            abi.iptr(rows))
    assert rc == 0, rc
    return np.swapaxes(Cb, -1, -2), int(rows[0])


def probe_potrf(Ms, mode=1, mask=None, L0=None, X0=None, info0=None):
    """Ms (nb, n, n) symmetric.  Returns the output buffers (L with the factor in its lower triangle, invdiag as
    (nb, nblk, 128, 128) natural blocks) and info.  L0 / X0 / info0 preset the buffers (what masked instances must keep)."""
    nb, n, _ = Ms.shape
    Lb = _colmajor(Ms if L0 is None else L0)
    Xb = np.ascontiguousarray(np.zeros((nb, n // NB, NB, NB)) if X0 is None else np.swapaxes(X0, -1, -2))
    info = np.zeros(nb, np.int64) if info0 is None else _ints(info0).copy()
    mk = _ints(mask)
    rc = _lib().qpalm_b200_dense_probe_potrf(nb, n, abi.fptr(Lb), abi.fptr(Xb), _iptr(mk), abi.iptr(info), mode)
    assert rc == 0, rc
    return np.swapaxes(Lb, -1, -2), np.swapaxes(Xb, -1, -2), info


def probe_trtri(L):
    n = len(L)
    Xb = np.zeros((n // NB, NB, NB))
    rc = _lib().qpalm_b200_dense_probe_trtri(n, abi.fptr(_colmajor(L[None])), abi.fptr(Xb))
    assert rc == 0, rc
    return np.swapaxes(Xb, -1, -2)


def probe_solve(L, X, V, mode, sizes=None, mask=None, Lbuf=None):
    """L (nb, n, n), X (nb, nblk, 128, 128), V (nb, rounds, n).  Round r solves the leading sizes[r] rows of V[:, r] with the
    leading block of L.  Lbuf: the column-major buffer of L itself (nb = 1), to spare a copy of a large L."""
    nb, rounds, n = V.shape
    Lb = _colmajor(L) if Lbuf is None else Lbuf
    Xb = np.ascontiguousarray(np.swapaxes(X, -1, -2))
    Vb = np.ascontiguousarray(V, dtype=np.float64).copy()
    sz, mk, grid = _ints(sizes), _ints(mask), np.zeros(rounds, np.int64)
    rc = _lib().qpalm_b200_dense_probe_solve(nb, n, abi.fptr(Lb), abi.fptr(Xb), abi.fptr(Vb), rounds, _iptr(sz), _iptr(mk), mode,
                                             abi.iptr(grid))
    assert rc == 0, rc
    return Vb, grid


# ------------------------------------------------------------------------------------------------
# references and bounds
# ------------------------------------------------------------------------------------------------
def check_gemm(Cg, A, B, C0, alpha, beta, what, sel=None):
    """Real data: every entry is beta c0 + alpha sum_k a_ik b_jk, DMMA chains in k order plus one multiply-add, so
    |C - C_exact| <= gamma_{K+2} (|A||B|' + |beta||C0|) (Higham Thm 3.5; |alpha| = 1 here), and the float64 reference formed
    here carries the same bound: 2 gamma_{K+2} for the difference.  sel: the entries to check (default all)."""
    K = A.shape[1]
    ref = beta * C0 + alpha * (A @ B.T)
    tol = 2 * gamma(K + 2) * (np.abs(A) @ np.abs(B).T + abs(beta) * np.abs(C0))
    err = np.abs(Cg - ref)
    if sel is not None:
        err, tol = err[sel], tol[sel]
    assert np.all(err <= tol), (what, float(np.max(err / np.maximum(tol, 1e-300))))
    return float(np.max(err / np.maximum(tol, 1e-300)))


def inverse_bound(Lb, Xb):
    """Bound on |L_bb X_bb - I| for the diagonal-block kernel's inverse.  Each 32 x 32 diagonal inverse is a column-wise forward
    substitution (Higham Thm 8.5 for every column: |L X - I| <= gamma_32 |L||X|).  Block row kb is then X(kb, <r0) =
    -X(kb,kb) R with R = L(kb, <r0) X(<r0, <r0) (R: sums of at most 100 products, X: of 32), so the residual of that block
    row is -E1 - (L_kk X_kk - I) R - L_kk E2 with |E1| <= gamma_100 |L||X|, |E2| <= gamma_32 |X_kk||R|: in all
    |L X - I| <= gamma_128 (|L||X| + 2 |L||X||L||X|)."""
    LX = np.abs(Lb) @ np.abs(Xb)
    return gamma(NB) * (LX + 2 * LX @ LX)


def check_inverse(Lb, Xb, what):
    """X_bb against its own factor block: the bound of inverse_bound twice over, plus gamma_128 |L||X| for the product formed
    here.  The upper triangle must be exactly zero (the solves read the full block)."""
    assert not np.any(np.triu(Xb, 1)), what
    res = np.abs(Lb @ Xb - np.eye(len(Lb)))
    tol = 2 * inverse_bound(Lb, Xb) + gamma(NB) * np.abs(Lb) @ np.abs(Xb)
    assert np.all(res <= tol), (what, float(np.max(res / np.maximum(tol, 1e-300))))


def factor_bound(L, X):
    """Entrywise bound on |L L' - M| for the blocked Cholesky.  The trailing updates (DMMA GEMMs, in-block FMA tiles) and the
    32-column in-register factorisations are Cholesky's standard recurrence in some order: gamma_{n+1} |L||L'| (Higham
    Thm 10.3).  The panels are different: L21 = fl(A21 X11') with X11 the computed inverse of the diagonal block (width w =
    32 inside the diagonal-block kernel, 128 for the in-place GEMM below it), so
        L21 L11' - A21 = A21 (X11' L11' - I) + E L11',  |E| <= gamma_w |A21||X11'|,
    i.e. |A21| (|L11 X11 - I|' + gamma_w |X11'||L11'|) on the panel's entries, with A21 ~ L21 L11' to first order.  For
    w = 128 |L11 X11 - I| is inverse_bound; for the 32 x 32 forward substitution it is gamma_32 |L11||X11|, X11 = inv(L11)
    formed here in float64 (first order)."""
    n = len(L)
    aL = np.abs(L)
    tol = gamma(n + 1) * (aL @ aL.T)
    for p in range(n // NB):
        s = slice(p * NB, (p + 1) * NB)
        Lpp, Xpp = aL[s, s], np.abs(X[p])
        if p * NB + NB < n:
            A21 = aL[(p + 1) * NB:, s] @ Lpp.T
            tol[(p + 1) * NB:, s] += A21 @ (inverse_bound(L[s, s], X[p]).T + gamma(NB) * Xpp.T @ Lpp.T)
        for q in range(3):
            c = slice(p * NB + 32 * q, p * NB + 32 * q + 32)
            r = slice(p * NB + 32 * q + 32, (p + 1) * NB)
            L32 = L[c, c]
            X32 = np.abs(np.linalg.inv(L32))
            A21 = aL[r, c] @ np.abs(L32).T
            tol[r, c] += gamma(32) * A21 @ (np.abs(L32) @ X32 + X32 @ np.abs(L32)).T
    return tol


def check_factor(L, X, M, what):
    """|L L' - M| <= 4 factor_bound: the first-order terms and the float64 rounding of L L' formed here (gamma_n |L||L'|)
    fit in the factor 4, a wrong entry of relative size 1e-12 does not (see the negative controls)."""
    assert np.all(np.diag(L) > 0), what
    err = np.abs(L @ L.T - M)
    tol = 4 * factor_bound(L, X)
    assert np.all(np.tril(err) <= np.tril(tol)), (what, float(np.max(np.tril(err) / np.maximum(np.tril(tol), 1e-300))))
    return float(np.max(np.tril(err) / np.maximum(np.tril(tol), 1e-300)))


def check_forward(L, M, X, kappa, norm2, what):
    """Forward error against LAPACK's factor.  Both factors are exact for a perturbed M: ours for |dM| <= 4 factor_bound,
    LAPACK's for |dM| <= 4 gamma_{n+1} |L||L'|.  Sun's first-order bound ||dL||_F <= kappa ||dM||_F / sqrt(||M||_2) (with
    ||L||_2 = sqrt(||M||_2)) for each, taken twice over."""
    Lref = np.linalg.cholesky(M)
    dM = np.linalg.norm(4 * factor_bound(L, X)) + np.linalg.norm(4 * gamma(len(L) + 1) * np.abs(Lref) @ np.abs(Lref).T)
    tol = 2 * kappa * dM / np.sqrt(norm2)
    err = np.max(np.abs(L - Lref))
    assert err <= tol, (what, err, tol)


def _amv(M, v, chunk=4096):
    """|M| v without a full |M| temporary."""
    return np.concatenate([np.abs(M[i:i + chunk]) @ v for i in range(0, M.shape[0], chunk)])


def solve_bound(L, X, x, b):
    """Bound on |b - L (L' x)| for x = chol_solve(b).  Forward, block i: t_i = b_i - sum_{j<i} L_ij y_j (|f| <=
    gamma_n (|b| + |L||y|)), y_i = fl(X_ii t_i) = X_ii t_i + e (|e| <= gamma_128 |X_ii||t_i|), so L_ii y_i + sum L_ij y_j - b_i
    = (L_ii X_ii - I) t_i + L_ii e + f.  Backward, block j: z_j = y_j - sum_{i>j} L_ij' x_i, x_j = X_jj' z_j + e', whose
    residual is (X_jj L_jj - I)' z_j + L_jj' e' + f', with the left residual |X L - I| <= |X| inverse_bound |L| to first
    order.  With L y = b + r_f and L' x = y + r_b, L L' x - b = r_f + L r_b.  First order: y ~ L' x, t_i ~ L_ii y_i,
    z_j ~ L_jj' x_j."""
    n = len(x)
    ax, ab = np.abs(x), np.abs(b)
    y = L.T @ x
    ay = np.abs(y)
    Bf = gamma(n) * (ab + _amv(L, ay))
    Bb = gamma(n) * (ay + _amv(L.T, ax))
    for k in range(n // NB):
        s = slice(k * NB, (k + 1) * NB)
        Lb, Xb = np.abs(L[s, s]), np.abs(X[k])
        t = Lb @ ay[s]
        LXt = Lb @ (Xb @ t)
        Bf[s] += gamma(NB) * (LXt + 2 * Lb @ (Xb @ LXt)) + gamma(NB) * LXt
        w = Xb.T @ (Lb.T @ ax[s])
        XLw = Xb.T @ (Lb.T @ w)
        Bb[s] += Lb.T @ (gamma(NB) * (XLw + 2 * Xb.T @ (Lb.T @ XLw))) + gamma(NB) * Lb.T @ w
    return Bf + _amv(L, Bb)


def check_solve(x, b, L, X, what):
    """|b - L L' x| <= 2 solve_bound (twice the first-order bound) + gamma_{2n+2} (|L||L'||x| + |b|) for the residual formed
    here."""
    n = len(x)
    assert np.all(np.isfinite(x)), what
    r = np.abs(b - L @ (L.T @ x))
    tol = 2 * solve_bound(L, X, x, b) + gamma(2 * n + 2) * (_amv(L, _amv(L.T, np.abs(x))) + np.abs(b))
    assert np.all(r <= tol), (what, float(np.max(r / tol)))
    return float(np.max(r / tol))


def graded(rng, n, cond):
    """spd(cond) scaled by D = 10^(-2 (i mod 128) / 127) on both sides: every 128 x 128 diagonal block has a condition number of
    about 1e4 times that of spd's blocks."""
    d = 10.0 ** (-2.0 * (np.arange(n) % NB) / (NB - 1))
    return d[:, None] * spd(rng, n, cond) * d[None, :]


def diag_dominant_factor(rng, n):
    """A lower-triangular factor built directly (no CPU factorisation): diagonal in [1, 2], strictly lower uniform(-1, 1) / n, so
    every row is diagonally dominant and the solves are well conditioned."""
    L = np.tril(rng.uniform(-1.0, 1.0, (n, n)) / n, -1)
    L[np.diag_indices(n)] = rng.uniform(1.0, 2.0, n)
    return L


# ------------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------------
GEMM_MN = (128, 256, 384, 1152)
GEMM_K = (16, 32, 48, 64, 80, 512, 4096)
AB = [(1.0, 0.0), (-1.0, 1.0), (1.0, 0.5), (-1.0, 0.0), (1.0, 1.0), (-1.0, 0.5)]


def _int_mat(rng, *shape):
    return rng.integers(-8, 9, shape).astype(np.float64)


def _expected(A, B, C0, alpha, beta, lower_only):
    ref = beta * C0 + alpha * (A @ B.T)
    if lower_only:
        M, N = C0.shape
        ti, tj = np.arange(M)[:, None] // NB, np.arange(N)[None, :] // NB
        ref = np.where(tj > ti, C0, ref)
    return ref


@gpu
@pytest.mark.parametrize("M", GEMM_MN)
def test_gemm_integer_exact(M):
    """Integer entries in [-8, 8], K <= 4096: every partial sum is an integer below 2^53, so the result is exact and must equal
    the float64 product bit for bit, for every (M, N, K) of the grid, all six (alpha, beta) pairs over the K values and
    lower_only on every other K (tiles strictly above the diagonal keep their input bits, diagonal tiles are fully written)."""
    rng = np.random.default_rng(10 + M)
    for N in GEMM_MN:
        for i, K in enumerate(GEMM_K):
            alpha, beta = AB[(i + N // NB) % len(AB)]
            lower = (i + N // NB) % 2 == 1
            A, B, C0 = _int_mat(rng, 1, M, K), _int_mat(rng, 1, N, K), _int_mat(rng, 1, M, N)
            Cg, _ = probe_gemm(A, B, C0, alpha, beta, lower_only=lower)
            assert np.array_equal(Cg[0], _expected(A[0], B[0], C0[0], alpha, beta, lower)), (M, N, K, alpha, beta, lower)


@gpu
def test_gemm_per_instance_k_mask_and_early_exit():
    """Per-instance Kz (0, 16, ..., K - 16) with nonzero data beyond Kz[b] that must not be read; masked instances unchanged;
    K = 0 with beta = 1 returns before writing (a -0.0 in C survives, which beta c + alpha 0 would turn into +0.0), K = 0 with
    beta != 1 scales C."""
    rng = np.random.default_rng(20)
    M, N, K = 384, 256, 512
    kz = [0, 16, 32, 48, 80, 256, 496, 0, 16, 480]
    mask = [1, 1, 1, 0, 1, 1, 1, 1, 0, 1]
    nb = len(kz)
    A, B, C0 = _int_mat(rng, nb, M, K), _int_mat(rng, nb, N, K), _int_mat(rng, nb, M, N)
    for alpha, beta in ((1.0, 1.0), (-1.0, 0.5), (1.0, 0.0)):
        for lower in (False, True):
            Cg, _ = probe_gemm(A, B, C0, alpha, beta, Kz=kz, mask=mask, lower_only=lower)
            for b in range(nb):
                k = kz[b]
                ref = C0[b] if not mask[b] else _expected(A[b, :, :k], B[b, :, :k], C0[b], alpha, beta, lower)
                assert np.array_equal(Cg[b], ref), (b, k, mask[b], alpha, beta, lower)
    Z = np.full((2, 128, 128), -0.0)
    for beta in (1.0, 0.5):
        Cg, _ = probe_gemm(np.zeros((2, 128, 0)), np.zeros((2, 128, 0)), Z, 1.0, beta)
        assert np.all(Cg == 0) and np.all(np.signbit(Cg) == (beta == 1.0)), beta
    Cg, _ = probe_gemm(np.zeros((1, 128, 0)), np.zeros((1, 128, 0)), C0[:1, :128, :128], -1.0, 0.5)
    assert np.array_equal(Cg[0], 0.5 * C0[0, :128, :128])
    Cg, _ = probe_gemm(A[:2], B[:2], np.full((2, M, N), -0.0), 1.0, 1.0, Kz=[0, 0])
    assert np.all(np.signbit(Cg))


@gpu
@pytest.mark.parametrize("M", [128, 1152])
def test_gemm_in_place(M):
    """C aliases A (the Cholesky's panel solve L21 <- L21 X'): N = 128, K = 128 and K = 64, beta 0 and 1, and a batch with a
    mask; each CTA waits for all its bulk copies before writing, so the result is exact."""
    rng = np.random.default_rng(30 + M)
    nb = 3
    C0, B = _int_mat(rng, nb, M, 128), _int_mat(rng, nb, 128, 128)
    for K in (128, 64):
        for alpha, beta in ((1.0, 0.0), (-1.0, 1.0)):
            Cg, _ = probe_gemm(None, B[:, :, :K], C0, alpha, beta, mask=[1, 0, 1], in_place=True)
            for b in range(nb):
                ref = C0[b] if b == 1 else beta * C0[b] + alpha * (C0[b, :, :K] @ B[b, :, :K].T)
                assert np.array_equal(Cg[b], ref), (M, K, alpha, beta, b)


@gpu
@pytest.mark.parametrize("K", [16, 80, 512, 4096])
def test_gemm_real_bound_and_both_tile_kernels(K):
    """Random real entries against the gamma_{K+2} bound of check_gemm; then the same instance once alone (fewer tiles than SMs:
    the 64-row kernel) and as SMs copies (the 128-row kernel): each entry runs the same k-ordered DMMA chain in both, so the
    bits are identical.  Full and lower_only shapes."""
    rng = np.random.default_rng(40 + K)
    sms = _sms()
    for M, N, lower in ((128, 128, False), (384, 384, True), (1152, 128, False)):
        A, B = rng.standard_normal((1, M, K)), rng.standard_normal((1, N, K))
        C0 = rng.standard_normal((1, M, N))
        for alpha, beta in ((1.0, 1.0), (-1.0, 0.5)):
            C1, rows1 = probe_gemm(A, B, C0, alpha, beta, lower_only=lower)
            tiles = (M // NB) * (N // NB) if not lower else (M // NB) * (M // NB + 1) // 2
            assert tiles < sms and rows1 == 64, (M, N, rows1)
            above = np.arange(N)[None, :] // NB > np.arange(M)[:, None] // NB
            if lower:
                assert np.array_equal(C1[0][above], C0[0][above])
            check_gemm(C1[0], A[0], B[0], C0[0], alpha, beta, (M, N, K, lower), sel=~above if lower else None)
            nb = -(-sms // tiles)
            Cn, rowsn = probe_gemm(np.repeat(A, nb, 0), np.repeat(B, nb, 0), np.repeat(C0, nb, 0), alpha, beta, lower_only=lower)
            assert rowsn == 128, (M, N, nb, rowsn)
            for b in range(nb):
                assert np.array_equal(Cn[b], C1[0]), (M, N, K, b)


# ------------------------------------------------------------------------------------------------
# factorisation and trtri
# ------------------------------------------------------------------------------------------------
FACTOR_NPAD = (128, 256, 384, 512, 640, 1024, 1152, 1664, 2560)


def _factor_cases(rng, n):
    """(name, M, kappa, ||M||_2): condition numbers 1e1 and 1e8 with a known spectrum, and a graded matrix whose diagonal
    blocks are ill-conditioned themselves (its kappa from the eigenvalues)."""
    out = [(f"cond{c:.0e}", spd(rng, n, c), c, 2.5) for c in (1e1, 1e8)]
    if n <= 1152:
        G = graded(rng, n, 1e2)
        ev = np.linalg.eigvalsh(G)
        out.append(("graded", G, ev[-1] / ev[0], ev[-1]))
    return out


@gpu
@pytest.mark.parametrize("npad", FACTOR_NPAD)
def test_factor_trtri_and_solves(npad):
    """potrf_lower (mode 0: the look-ahead above 1024) on each case: L against factor_bound and against LAPACK's factor, each
    invdiag block against its own L block (check_inverse), trtri_diag_blocks on the returned L bit-identical to the invdiag
    the factorisation wrote; then both solves (mode 0: the dataflow solve above 256; mode 1: the per-block launches) for three
    different right-hand sides in three rounds on one stream."""
    rng = np.random.default_rng(50 + npad)
    for name, M, kappa, norm2 in _factor_cases(rng, npad):
        what = (npad, name)
        L, X, info = probe_potrf(M[None], mode=0)
        L, X = np.tril(L[0]), X[0]
        assert info[0] == 0, what
        check_factor(L, X, M, what)
        check_forward(L, M, X, kappa, norm2, what)
        for k in range(npad // NB):
            s = slice(k * NB, (k + 1) * NB)
            check_inverse(L[s, s], X[k], what + (k,))
        assert np.array_equal(probe_trtri(L), X), what
        rhs = rng.standard_normal((1, 3, npad)) * np.array([1.0, 1e3, 1e-3])[None, :, None]
        for mode in (0, 1):
            V, grid = probe_solve(L[None], X[None], rhs, mode)
            assert np.all(grid == (min(npad // NB, _sms()) if mode == 0 and npad > 2 * NB else 0)), (what, mode, grid)
            for r in range(3):
                check_solve(V[0, r], rhs[0, r], L, X, what + (mode, r))


@gpu
def test_factor_large():
    """npad = 4096 (3 look-ahead rounds with the rest update carried over 512-column outer blocks 4 times), M = B B' / n + I:
    kappa <= ||M||_inf (the eigenvalues are >= 1); factor, inverse and dataflow solve as above."""
    n = 4096
    rng = np.random.default_rng(60)
    Bm = rng.standard_normal((n, n))
    M = Bm @ Bm.T / n + np.eye(n)
    L, X, info = probe_potrf(M[None], mode=0)
    L, X = np.tril(L[0]), X[0]
    assert info[0] == 0
    check_factor(L, X, M, "n4096")
    norm_inf = np.max(np.sum(np.abs(M), axis=1))
    check_forward(L, M, X, norm_inf, np.max(np.diag(M)), "n4096")
    for k in range(n // NB):
        s = slice(k * NB, (k + 1) * NB)
        check_inverse(L[s, s], X[k], ("n4096", k))
    rhs = rng.standard_normal((1, 3, n))
    V, grid = probe_solve(L[None], X[None], rhs, 0)
    assert np.all(grid > 0)
    for r in range(3):
        check_solve(V[0, r], rhs[0, r], L, X, ("n4096", r))


@gpu
@pytest.mark.parametrize("npad", [1152, 1664, 2560])
def test_lookahead_schedule_is_bit_identical(npad):
    """The look-ahead (mode 0: 1, 2 and 3 rounds at these sizes) splits each rank-512 update into the next block's first slab,
    its other slabs on a second stream, and the rest, in other launches than the batched schedule's single update (mode 1
    with nb = 1).  Each entry still receives the same k-ordered DMMA chains and the same diagonal-block kernel runs: L, invdiag
    and info are bit-identical."""
    rng = np.random.default_rng(70 + npad)
    M = spd(rng, npad, 1e4)
    L0, X0, i0 = probe_potrf(M[None], mode=0)
    L1, X1, i1 = probe_potrf(M[None], mode=1)
    assert i0[0] == i1[0] == 0
    assert np.array_equal(np.tril(L0), np.tril(L1))
    assert np.array_equal(X0, X1)


def _indefinite(rng, n, col):
    """L0 D L0' with D = I except D[col, col] = -1: leading minors of order <= col are those of an SPD matrix, the pivot at
    col is -L0[col, col]^2."""
    L0 = np.linalg.cholesky(base(rng, n))
    d = np.ones(n)
    d[col] = -1.0
    return (L0 * d) @ L0.T


@gpu
@pytest.mark.parametrize("npad", [256, 640])
def test_batched_factor_masks_and_pivots(npad):
    """nb = 2 SMs + 3 instances (npad = 640 crosses the 512-column outer block): seven different SPD matrices in turn, every
    fifth instance masked (L, invdiag and info keep their input bits), and instances whose first non-positive pivot sits at
    column c in {0, 31, 32, 127, 128, 511, 512, 600} (info = c + 1).  Every copy of a matrix is bit-identical to the others and
    to the nb = 1 run of the batched schedule, which is checked against the bounds."""
    rng = np.random.default_rng(80 + npad)
    nb = 2 * _sms() + 3
    mats = [spd(rng, npad, c) for c in (1e1, 1e3, 1e8, 1e2, 1e5, 1e1, 1e6)]
    cols = [c for c in (0, 31, 32, 127, 128, 511, 512, 600) if c < npad]
    bad = [_indefinite(rng, npad, c) for c in cols]
    kind = []
    for b in range(nb):
        if b % 5 == 4:
            kind.append(("masked", b % 7))
        elif b % 11 == 3 and len([k for k in kind if k[0] == "bad"]) < len(cols):
            kind.append(("bad", len([k for k in kind if k[0] == "bad"])))
        else:
            kind.append(("ok", b % 7))
    for c in range(len(cols)):   # every pivot column appears (the loop above places them while instances last)
        assert ("bad", c) in kind
    mask = [0 if k == "masked" else 1 for k, _ in kind]
    L0 = rng.standard_normal((nb, npad, npad))          # masked instances keep this
    for b, (k, i) in enumerate(kind):
        if k != "masked":
            L0[b] = bad[i] if k == "bad" else mats[i]
    X0 = rng.standard_normal((nb, npad // NB, NB, NB))
    info0 = np.where(np.array(mask) == 0, 7, 0)
    Lfull, X, info = probe_potrf(L0, mode=1, mask=mask, L0=L0, X0=X0, info0=info0)
    singles = {}
    for i, M in enumerate(mats):
        Ls, Xs, inf = probe_potrf(M[None], mode=1)
        assert inf[0] == 0
        check_factor(np.tril(Ls[0]), Xs[0], M, (npad, "single", i))
        singles[i] = (np.tril(Ls[0]), Xs[0])
    for b, (k, i) in enumerate(kind):
        if k == "masked":
            assert np.array_equal(Lfull[b], L0[b]) and np.array_equal(X[b], X0[b]) and info[b] == 7, b
        elif k == "bad":
            assert info[b] == cols[i] + 1, (b, cols[i], info[b])
        else:
            assert info[b] == 0, b
            assert np.array_equal(np.tril(Lfull[b]), singles[i][0]) and np.array_equal(X[b], singles[i][1]), (b, i)


@gpu
def test_lookahead_pivot_after_a_lookahead_round():
    """Mode 0 at npad = 1152: the first non-positive pivot at column 1000, in the last outer block after one look-ahead round.
    L0 D L0' and L0 L0' agree bit for bit in every column before 1000 (numpy adds the same products), so the factor's columns
    before the pivot's diagonal block (896) match the healthy matrix's factor bit for bit."""
    rng = np.random.default_rng(90)
    n, col = 1152, 1000
    L0 = np.linalg.cholesky(base(rng, n))
    d = np.ones(n)
    d[col] = -1.0
    M, Mh = (L0 * d) @ L0.T, L0 @ L0.T
    assert np.array_equal(M[:, :col], Mh[:, :col])
    L, X, info = probe_potrf(M[None], mode=0)
    Lh, Xh, infoh = probe_potrf(Mh[None], mode=0)
    assert info[0] == col + 1 and infoh[0] == 0, (info, infoh)
    assert np.array_equal(np.tril(L[0])[:, :896], np.tril(Lh[0])[:, :896])
    assert np.array_equal(X[0][:7], Xh[0][:7])


# ------------------------------------------------------------------------------------------------
# solves: batched with masks, rounds of different sizes, more blocks than the cooperative grid
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("npad", [256, 640, 1152])
def test_batched_solve_with_mask(npad):
    """chol_solve_batched over 5 instances, 3 rounds with different right-hand sides, instances 1 and 3 masked (their vectors
    keep their bits)."""
    rng = np.random.default_rng(100 + npad)
    nb = 5
    Ls = np.stack([np.linalg.cholesky(spd(rng, npad, 10.0 ** (b + 1))) for b in range(nb)])
    Xs = np.stack([probe_trtri(Ls[b]) for b in range(nb)])
    V0 = rng.standard_normal((nb, 3, npad))
    mask = [1, 0, 1, 0, 1]
    V, grid = probe_solve(Ls, Xs, V0, 1, mask=mask)
    assert not np.any(grid)
    for b in range(nb):
        for r in range(3):
            if mask[b]:
                check_solve(V[b, r], V0[b, r], Ls[b], Xs[b], (npad, b, r))
            else:
                assert np.array_equal(V[b, r], V0[b, r])


@gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_solve_rounds_of_growing_size(mode):
    """Rounds on one stream at sizes 384, 384, 4608, 4608, 1152, 640: the dataflow solve's packet ring grows (a ring of
    2 * nblk + 64 blocks is reallocated, the epoch restarts) and is reused at smaller sizes; each round solves the leading
    block of one directly built factor, entries beyond it untouched."""
    n = 4608
    rng = np.random.default_rng(110)
    L = diag_dominant_factor(rng, n)
    X = probe_trtri(L)
    sizes = [384, 384, 4608, 4608, 1152, 640]
    V0 = rng.standard_normal((1, len(sizes), n))
    V, grid = probe_solve(L[None], X[None], V0, mode, sizes=sizes)
    for r, m in enumerate(sizes):
        assert grid[r] == (min(m // NB, _sms()) if mode == 0 else 0), (r, grid)
        assert np.array_equal(V[0, r, m:], V0[0, r, m:])
        check_solve(V[0, r, :m], V0[0, r, :m], L[:m, :m], X[:m // NB], (mode, r, m))


def _mem_available():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


@gpu
def test_dataflow_solve_with_more_blocks_than_the_grid():
    """npad = 128 (grid + 2) with grid = SMs (one CTA per SM: 137 kB of shared memory each): CTAs 0 and 1 own two blocks each
    (c and c + grid) in both sweeps.  L is built directly (diagonal in [1, 2], strictly lower uniform(-1, 1) / n), its
    diagonal-block inverses by trtri_diag_blocks; three rounds."""
    import torch
    n = NB * (_sms() + 2)
    need = 8 * n * n
    if torch.cuda.mem_get_info()[0] < need + (1 << 30) or _mem_available() < 3 * need:
        pytest.skip("not enough device or host memory for a %d x %d factor" % (n, n))
    rng = np.random.default_rng(120)
    Lt = rng.uniform(-1.0, 1.0, (n, n))      # L' in C order: the column-major buffer of L
    Lt /= n
    for i in range(0, n, 1024):
        Lt[i:i + 1024] = np.triu(Lt[i:i + 1024], i + 1)
    Lt[np.diag_indices(n)] = rng.uniform(1.0, 2.0, n)
    L = Lt.T
    X = np.stack([np.linalg.inv(L[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB]) for k in range(n // NB)])
    X = np.where(np.tril(np.ones((NB, NB), bool)), X, 0.0)
    V0 = rng.standard_normal((1, 3, n))
    V, grid = probe_solve(None, X[None], V0, 0, Lbuf=Lt)
    assert np.all(grid == _sms()) and np.all(grid < n // NB), grid
    for r in range(3):
        check_solve(V[0, r], V0[0, r], L, X, ("nblk > grid", r))


# ------------------------------------------------------------------------------------------------
# solver level: the lock-step engine with npad = 640
# ------------------------------------------------------------------------------------------------
@gpu
def test_lockstep_engine_npad640_against_oracle():
    """n = 600, m = 1200: beyond the persistent engine, so the lock-step engine runs its batched Cholesky at npad = 640, where
    the rank-512 update of the last 128 columns runs with the live instance masks; every instance against the oracle."""
    nb = 5
    b = problems.mpc_batch(nb, n=600, m0=600, seed=51)
    h = qb.Batch(b.Q, b.A, b.settings, nb)
    assert h.ok
    xs, ys, infos = h.solve(b.q, b.bmin, b.bmax)
    shape = h.last_shape()
    h.cleanup()
    assert shape == 0
    _check_instances(b, range(nb), xs, ys, infos)


# ------------------------------------------------------------------------------------------------
# negative controls (no GPU): the checks reject results that are wrong by a little
# ------------------------------------------------------------------------------------------------
def _rejects(check, *args):
    with pytest.raises(AssertionError):
        check(*args)


def test_gemm_check_rejects_perturbed_entry_and_missing_k_tile():
    """At K = 16 and 64 a relative 1e-12 change of one entry is above gamma_{K+2} |A||B|' (at K = 4096 it is not: gamma_4098
    is 4.5e-13); one missing k-tile changes entries by O(sqrt(16)) times the inputs' size."""
    rng = np.random.default_rng(1)
    for K in (16, 64, 4096):
        A, B, C0 = rng.standard_normal((256, K)), rng.standard_normal((128, K)), rng.standard_normal((256, 128))
        C = 0.5 * C0 - A @ B.T
        check_gemm(C, A, B, C0, -1.0, 0.5, K)
        missing = C + A[:, K - 16:] @ B[:, K - 16:].T
        _rejects(check_gemm, missing, A, B, C0, -1.0, 0.5, K)
        if K <= 64:
            i, j = np.unravel_index(np.argmax(np.abs(C)), C.shape)
            bad = C.copy()
            bad[i, j] *= 1 + 1e-12
            _rejects(check_gemm, bad, A, B, C0, -1.0, 0.5, K)


def _host_factor(rng, n):
    M = base(rng, n)
    L = np.linalg.cholesky(M)
    X = np.stack([np.tril(np.linalg.inv(L[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB])) for k in range(n // NB)])
    return M, L, X


def test_factor_inverse_and_solve_checks_reject_perturbed_entries():
    """LAPACK's factor of a well-conditioned matrix, inv() of its diagonal blocks and a float64 solve pass the checks; one entry
    off by a relative 1e-12 fails them: L in the first block column (diagonal, inside the diagonal block, below it: the
    GEMM panel), X on its diagonal and at its largest entry below it, x at its largest entry (for a diagonally dominant
    factor)."""
    rng = np.random.default_rng(2)
    n = 256
    M, L, X = _host_factor(rng, n)
    check_factor(L, X, M, "host")
    for k in range(n // NB):
        check_inverse(L[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB], X[k], k)
    for i, j in ((0, 0), (100, 0), (200, 0), (255, 1)):
        bad = L.copy()
        bad[i, j] *= 1 + 1e-12
        _rejects(check_factor, bad, X, M, (i, j))
    off = np.unravel_index(np.argmax(np.abs(np.tril(X[0], -1))), X[0].shape)
    for i, j in ((5, 5), off):
        bad = X[0].copy()
        bad[i, j] *= 1 + 1e-12
        _rejects(check_inverse, L[:NB, :NB], bad, (i, j))
    # the solve bound sums |L||L'||x| over whole rows: a 1e-12 change of one component stands out of it where L is
    # diagonally dominant (for a dense factor of this size it is within the rounding of the other n - 1 terms)
    L = diag_dominant_factor(rng, n)
    X = np.stack([np.tril(np.linalg.inv(L[k * NB:(k + 1) * NB, k * NB:(k + 1) * NB])) for k in range(n // NB)])
    b = rng.standard_normal(n)
    x = np.linalg.solve(L.T, np.linalg.solve(L, b))
    check_solve(x, b, L, X, "host")
    bad = x.copy()
    k = int(np.argmax(np.abs(x)))
    bad[k] *= 1 + 1e-12
    _rejects(check_solve, bad, b, L, X, "perturbed")
