"""The dense factor's generator-form rank-k update / downdate (updown_gen.cu) against float64 references, stage by stage:

    k_fwd_multi                        What = inv(L) W                   (cooperative dataflow solve, Tdump running sums)
    k_gen_gram / k_gen_scan / k_gen_rows   M_B = S + What_<B' What_<B, d_j, z_j    (Gauss-Jordan + Sherman-Morrison per 32 rows)
    k_gen_apply                        L_new(r, j) = d_j L(r, j) + (W_r - sum_{i <= j} L(r, i) what_i)' z_j

through qpalm_b200_dense_probe_updown, which runs the production functions unchanged on caller data on one fresh stream, and
through the per-panel sweep of dense.cu (chol_updown) that the solver uses below two blocks.  The algebra is restated in numpy
by test_generator_update_math.generator_update.

Tolerances are a-priori rounding-error bounds with u = eps / 2 and gamma_k = k u / (1 - k u) (Higham, Accuracy and Stability
of Numerical Algorithms, 2nd ed.), evaluated on the GPU's own inputs and outputs, first order:

* What (check_what): block row i is t_i = W_i - sum_{j < i} L_ij What_j (DMMA sums, |f| <= gamma_n (|W| + |L||What|)), then
  What_i = fl(X_ii t_i) with X_ii the explicitly inverted diagonal block (|e| <= gamma_128 |X_ii||t_i|), so the residual
  W - L What of the block is (L_ii X_ii - I) t_i + L_ii e + f: test_gpu_dense.inverse_bound for the first term, twice over,
  plus gamma_n (|W| + |L||What|) for the residual formed here.
* D (check_dz): d^2 = 1 + what' g with g = P what (k products: gamma_k), d = sqrt correctly rounded, z = g / d with a rounded
  reciprocal: |d^2 - 1 - d what' z| <= 3 gamma_{k+4} (1 + d |what|'|z|), the factor 3 covering the evaluation here.
* Z (check_dz): g = d z must solve M_j g = what_j, M_j = S + sum_{p<j} what_p what_p' formed here from the returned What, P_j =
  inv(M_j).  The kernel's P is the Gauss-Jordan inverse of the scanned Gram prefix M_B of its 32-row block, updated by
  Sherman-Morrison steps.  An error dM of M_B moves P_j by -P_j dM P_j and an error dP_B of P_B by P_j M_B dP_B M_B P_j, so
  |M_j g - what_j| <= [ gamma_2k (|M_B||P_B| + (|M_B||P_B|)^2) |M_B| |P_j| + gamma_n |What_<B|'|What_<B| |P_j| ] |what_j|
  (Gauss-Jordan residual, Gram and scan sums) + gamma_{k+3} |M_j| sum_{B0 <= i < j} (|P_i| + |z_i||z_i|') |M_j| |g|
  (Sherman-Morrison roundings) + gamma_k |M_j||P_j||what_j| (g = P what) + gamma_n (|What_<j|'|What_<j| + I) |g| (M_j formed
  here); asserted at twice that.
* The updated factor (check_apply): the exact formula above from the returned What, Z, D.  The tile's running sum (Tdump, a
  DMMA sum) and the column-by-column updates of t: |dt| <= gamma_{j+2} (|W_r| + sum_{i <= j} |L(r, i)||what_i|); the output
  d l + t'z: gamma_{k+2} (d |l| + |t|'|z|) + |dt|'|z|; twice that for the same evaluation here.  A wrong Tdump tile start or
  a wrong diagonal-tile column limit (jmax) changes entries by O(|L||What||z|).
* End to end (check_residual): L_new L_new' against L L' + W S W'.  With K the unit-generator factor built from the returned
  generators (K_jj = d_j, K_ij = what_i' z_j), L_new = L K up to the stage errors above, each bounded by a gamma_{n+k+64}
  multiple of |L||K| (the growth of the product before cancellation) or of |L||L'| + |W||W'|; so
  |L_new L_new' - L L' - W S W'| <= 8 gamma_{n+k+64} (|L||K||K'||L'| + |L||L'| + |W||W'|).  A wrong sign of one column of
  S changes it by 2 |w w'|, far outside.  Where the bound does not apply (ill-conditioned M_j: the solver and near-singular
  families) the pass is compared with the oracle's restatement of CHOLMOD's recurrence on the same inputs instead: the GPU's
  normwise residual at most RATIO_MAX = 8 times the oracle's (for a mixed pass the oracle's update then its downdate).
* Forward error (check_forward): against LAPACK's factor of L L' + W S W' where that matrix is well conditioned; Sun's
  first-order bound kappa ||dH||_F / sqrt(||H||_2) for each factor's backward error, taken twice over.
* Failure reporting: k_gen_rows sets info = 1 + 32 B for a 32-row block B with a non-positive d_j^2 or pivot; blocks before
  the first failing row are exact, so info - 1 >= 32 floor(first failing row / 32).  info == 0 must come with a finite L.

The measured margins (error over bound) and GPU / oracle ratios are printed with -s.  The negative controls at the end run
without a GPU: each check rejects a result with one entry off by a relative 1e-12 where its bound is tight enough (the What,
D and apply checks; the end-to-end residual is summed over whole rows and cannot see it), one column with the wrong sign in S,
a Tdump tile start left at zero, and a mixed pass whose kpos is off by one."""
import ctypes as C

import numpy as np
import pytest

from qpalm_b200 import abi, problems
from qpalm_b200.interface import load_library
from test_gpu_batch_cta import base, spd
from test_gpu_dense import NB, _iptr, _ints, diag_dominant_factor, gamma, gpu, inverse_bound
from test_generator_update_math import generator_update

GB = 32
RATIO_MAX = 8.0
WIDTHS = (1, 7, 8, 9, 15, 16, 17, 24, 31, 32)
MARGINS = {}


def _note(key, v):
    MARGINS[key] = max(MARGINS.get(key, 0.0), float(v))
    print(f"[updown_gen] {key}: {float(v):.3g}")


# ------------------------------------------------------------------------------------------------
# probe
# ------------------------------------------------------------------------------------------------
def _lib():
    lib = load_library("b200")
    if not getattr(lib, "_updown_probe_typed", False):
        fp, ip, ci = abi.c_float_p, abi.c_int_p, abi.c_int
        lib.qpalm_b200_dense_probe_updown.argtypes = [ci, fp, fp, ci, ip, ip, ip, ci, ci, ip, ip, fp, fp, fp]
        lib.qpalm_b200_dense_probe_updown.restype = C.c_int
        lib._updown_probe_typed = True
    return lib


def probe_updown(L, Ws, kpos, sizes=None, mode=0, cap=0, stages=True, Lbuf=None):
    """Passes r = 0 .. on one stream: L L' += W_r S_r W_r' on the leading sizes[r] block.  L (npad x npad) or Lbuf (its
    column-major buffer, updated in place).  Returns (L_new, info, grid (passes x 2: grid that ran, its limit), What, Z, D of
    the last pass (rows of the last size))."""
    npad = len(L) if Lbuf is None else Lbuf.shape[0]
    Lb = np.ascontiguousarray(L.T) if Lbuf is None else Lbuf
    ks = [W.shape[1] for W in Ws]
    Wb = np.ascontiguousarray(np.hstack(Ws).T)
    info, grid = np.zeros(len(Ws), np.int64), np.zeros((len(Ws), 2), np.int64)
    kl = ks[-1]
    What, Z, D = (np.zeros((kl, npad)), np.zeros((kl, npad)), np.zeros(npad)) if stages else (None, None, None)
    rc = _lib().qpalm_b200_dense_probe_updown(npad, abi.fptr(Lb), abi.fptr(Wb), len(Ws), abi.iptr(_ints(ks)), abi.iptr(_ints(kpos)),
                                              _iptr(_ints(sizes)), mode, cap, abi.iptr(info), abi.iptr(grid),
                                              abi.fptr(What) if stages else None, abi.fptr(Z) if stages else None,
                                              abi.fptr(D) if stages else None)
    assert rc == 0, rc
    n = npad if sizes is None else sizes[-1]
    st = (What.T[:n].copy(), Z.T[:n].copy(), D[:n].copy()) if stages else (None, None, None)
    return (Lb.T if Lbuf is None else None), info, grid, st


def signs(k, kpos):
    return np.array([1.0] * kpos + [-1.0] * (k - kpos))


# ------------------------------------------------------------------------------------------------
# references and bounds
# ------------------------------------------------------------------------------------------------
def _margin(err, tol):
    return float(np.max(err / np.maximum(tol, 1e-300))) if err.size else 0.0


def check_what(Wh, L, W, what, rows=None):
    """W - L What against the dataflow solve's bound (module docstring); rows: the 128-row blocks to check (default all)."""
    n = len(L)
    blocks = range(n // NB) if rows is None else rows
    m = 0.0
    for b in blocks:
        s = slice(b * NB, (b + 1) * NB)
        Lr = L[s, :(b + 1) * NB]
        aW, aL = np.abs(W[s]), np.abs(Lr)
        Lb = L[s, s]
        Xb = np.tril(np.linalg.inv(Lb))
        res = np.abs(W[s] - Lr @ Wh[:(b + 1) * NB])
        t = np.abs(Lb) @ np.abs(Wh[s])
        LXt = np.abs(Lb) @ (np.abs(Xb) @ t)
        tol = 2 * (inverse_bound(Lb, Xb) @ t + gamma(NB) * LXt) + 3 * gamma(n + 1) * (aW + aL @ np.abs(Wh[:(b + 1) * NB]))
        assert np.all(res <= tol), (what, "What", b, _margin(res, tol))
        m = max(m, _margin(res, tol))
    return m


def _prefix(Wh, sg):
    """M_j = S + sum_{p<j} what_p what_p' for every row j, and the element-wise |What|'|What| prefix."""
    n, k = Wh.shape
    outer = Wh[:, :, None] * Wh[:, None, :]
    M = np.cumsum(outer, axis=0) - outer + np.diag(sg)[None]
    A = np.cumsum(np.abs(outer), axis=0) - np.abs(outer)
    return M, A


def check_dz(Wh, Z, D, kpos, what):
    """d and z of k_gen_rows against their consistency with What (module docstring)."""
    n, k = Wh.shape
    sg = signs(k, kpos)
    u1 = np.abs(D ** 2 - 1.0 - D * np.sum(Wh * Z, axis=1))
    t1 = 3 * gamma(k + 4) * (1.0 + D * np.sum(np.abs(Wh) * np.abs(Z), axis=1))
    assert np.all(np.isfinite(D)) and np.all(D > 0), what
    assert np.all(u1 <= t1), (what, "d", int(np.argmax(u1 / t1)), _margin(u1, t1))
    M, A = _prefix(Wh, sg)
    P = np.linalg.inv(M)
    aM, aP = np.abs(M), np.abs(P)
    g = D[:, None] * Z
    res = np.abs(np.einsum("jab,jb->ja", M, g) - Wh)
    aw, ag = np.abs(Wh), np.abs(g)
    tol = np.zeros_like(res)
    for b0 in range(0, n, GB):
        MB, PB, AB = aM[b0], aP[b0], A[b0]
        MP = MB @ PB
        GJ = gamma(2 * k) * (MP + MP @ MP) @ MB
        acc = np.zeros((k, k))
        for j in range(b0, min(n, b0 + GB)):
            tol[j] = (GJ @ (aP[j] @ aw[j]) + gamma(n) * AB @ (aP[j] @ aw[j]) + gamma(k + 3) * aM[j] @ (acc @ (aM[j] @ ag[j]))
                      + gamma(k) * aM[j] @ (aP[j] @ aw[j]) + gamma(n) * (A[j] + np.eye(k)) @ ag[j])
            acc += aP[j] + np.outer(np.abs(Z[j]), np.abs(Z[j]))
    tol *= 2
    assert np.all(res <= tol), (what, "z", int(np.argmax(np.max(res / np.maximum(tol, 1e-300), axis=1))), _margin(res, tol))
    return max(_margin(u1, t1), _margin(res, tol))


def check_apply(Lg, L, W, Wh, Z, D, what, rows=None, tile_start_zero=False):
    """L_new from the exact formula on the GPU's What, Z, D (module docstring).  rows: row indices to check (default all).
    tile_start_zero: the negative control's reference with every Tdump tile start left at zero."""
    n, k = W.shape
    rows = np.arange(n) if rows is None else np.asarray(rows)
    Lr, Wr = L[rows], W[rows]
    T = Wr.copy()
    A = np.abs(Wr).copy()
    ref, tol = np.zeros((len(rows), n)), np.zeros((len(rows), n))
    for j in range(n):
        if tile_start_zero and j % NB == 0 and j > 0:
            T = Wr.copy()
        l = Lr[:, j]
        T -= l[:, None] * Wh[j][None, :]
        A += np.abs(l)[:, None] * np.abs(Wh[j])[None, :]
        ref[:, j] = D[j] * l + T @ Z[j]
        az = np.abs(Z[j])
        tol[:, j] = 2 * (gamma(k + 2) * (D[j] * np.abs(l) + np.abs(T) @ az) + gamma(j + 2) * A @ az)
    low = rows[:, None] >= np.arange(n)[None, :]
    err = np.where(low, np.abs(Lg[rows] - ref), 0.0)
    tol = np.where(low, tol, 1.0)
    assert np.all(err <= tol), (what, "apply", np.unravel_index(np.argmax(err / tol), err.shape), _margin(err, tol))
    return _margin(err, tol)


def k_factor(Wh, Z, D):
    K = np.tril(Wh @ Z.T, -1)
    K[np.diag_indices(len(D))] = D
    return K


def check_residual(Lg, L, W, kpos, Wh, Z, D, what, rows=None):
    """|L_new L_new' - (L L' + W S W')| <= 8 gamma_{n+k+64} (|L||K||K'||L'| + |L||L'| + |W||W'|) on the given rows."""
    n, k = W.shape
    rows = np.arange(n) if rows is None else np.asarray(rows)
    sg = signs(k, kpos)
    Lg = np.tril(Lg)
    H = L[rows] @ L.T + (W[rows] * sg) @ W.T
    res = np.abs(Lg[rows] @ Lg.T - H)
    aL = np.abs(L)
    LK = aL @ np.abs(k_factor(Wh, Z, D))
    tol = 8 * gamma(n + k + 64) * (LK[rows] @ LK.T + aL[rows] @ aL.T + np.abs(W[rows]) @ np.abs(W).T)
    assert np.all(res <= tol), (what, "residual", np.unravel_index(np.argmax(res / tol), res.shape), _margin(res, tol))
    return _margin(res, tol)


def normwise_residual(Lx, L, W, kpos):
    sg = signs(W.shape[1], kpos)
    Lx = np.tril(Lx)
    return float(np.max(np.abs(Lx @ Lx.T - L @ L.T - (W * sg) @ W.T)))


def oracle_pass(oracle_ops, L, W, kpos):
    """CHOLMOD's recurrence as the reference runs it: the update, then the downdate."""
    Lo = L
    if kpos > 0:
        Lo = oracle_ops.updown(Lo, W[:, :kpos], 1)
    if kpos < W.shape[1]:
        Lo = oracle_ops.updown(Lo, W[:, kpos:], 0)
    return Lo


def check_against_oracle(Lg, L, W, kpos, oracle_ops, what, family):
    """The GPU's normwise residual at most RATIO_MAX times the oracle's (floored at one rounding of the largest entry)."""
    Lo = oracle_pass(oracle_ops, L, W, kpos)
    rg, ro = normwise_residual(Lg, L, W, kpos), normwise_residual(Lo, L, W, kpos)
    floor = gamma(1) * float(np.max(np.abs(L) @ np.abs(L).T + np.abs(W) @ np.abs(W).T))
    ratio = rg / max(ro, floor)
    _note(f"oracle ratio {family}", ratio)
    assert ratio <= RATIO_MAX, (what, rg, ro, ratio)
    return ratio


def check_forward(Lg, L, W, kpos, what):
    sg = signs(W.shape[1], kpos)
    H = L @ L.T + (W * sg) @ W.T
    ev = np.linalg.eigvalsh(H)
    Lr = np.linalg.cholesky(H)
    n = len(L)
    dH = np.linalg.norm(np.abs(Lg @ Lg.T - H)) + np.linalg.norm(4 * gamma(n + 1) * np.abs(Lr) @ np.abs(Lr).T)
    dH = max(dH, np.linalg.norm(8 * gamma(n + W.shape[1] + 64) * (np.abs(L) @ np.abs(L).T + np.abs(W) @ np.abs(W).T)))
    tol = 2 * (ev[-1] / ev[0]) * dH / np.sqrt(ev[-1])
    err = np.max(np.abs(np.tril(Lg) - Lr))
    assert err <= tol, (what, "forward", err, tol)
    return err, tol


def check_valid(Lg, info, what):
    assert info == 0, (what, info)
    assert np.all(np.isfinite(np.tril(Lg))), what
    assert np.all(np.diag(Lg) > 0), what


def check_all(Lg, L, W, kpos, st, info, what, residual=True):
    """Every check of a valid pass: stages, end-to-end bound, validity; returns the margins."""
    check_valid(Lg, info, what)
    Wh, Z, D = st
    m = {"What": check_what(Wh, L, W, what), "D,Z": check_dz(Wh, Z, D, kpos, what), "apply": check_apply(Lg, L, W, Wh, Z, D, what)}
    if residual:
        m["residual"] = check_residual(Lg, L, W, kpos, Wh, Z, D, what)
    for key, v in m.items():
        _note("margin " + key, v)
    return m


def kpos_set(k):
    return sorted({0, 1, k // 2, k - 1, k} | {p for p in (7, 8, 9, 15, 16, 17) if p <= k})


def well_case(rng, n, k, kpos, zero_col=None):
    """base(n) plus the leaving columns (the downdate is valid on its own), entering columns of the same size."""
    W = rng.standard_normal((n, k))
    if zero_col is not None:
        W[:, zero_col] = 0.0
    H = base(rng, n) + W[:, kpos:] @ W[:, kpos:].T
    return np.linalg.cholesky(H), W


# ------------------------------------------------------------------------------------------------
# families
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", WIDTHS)
def test_well_conditioned_every_width_and_split(k):
    """Every KT / KW instantiation, pad columns and the second column group, with kpos on both sides of the 8- and 16-column
    group boundaries; npad 256 and 640 in turn (nblk 2 and 5).  Stages, end-to-end bound, forward error."""
    rng = np.random.default_rng(1000 + k)
    for i, kpos in enumerate(kpos_set(k)):
        n = 256 if i % 2 == 0 else 640
        L, W = well_case(rng, n, k, kpos)
        Lg, info, grid, st = probe_updown(L, [W], [kpos])
        what = ("well", n, k, kpos)
        check_all(Lg, L, W, kpos, st, info[0], what)
        err, tol = check_forward(Lg, L, W, kpos, what)
        _note("margin forward", err / tol)
        assert grid[0, 0] == min(n // NB, grid[0, 1]) > 0, (what, grid)


def solver_case(rng, n, beta, kind, k=32):
    """H = Q + A_J' Sigma_J A_J + beta I as QPALM forms it (sigma log-uniform in [1e-1, 1e8], |J| = 1.5 n so H stays definite
    after the leaving rows go); W = sqrt(sigma_i) a_i of entering rows (not in J, sign +1) and leaving rows (in J, sign -1)."""
    m = 3 * n
    A = rng.standard_normal((m, n)) * (rng.random((m, n)) < 0.2)
    Mq = rng.standard_normal((n, n // 4)) / np.sqrt(n)
    sig = 10.0 ** rng.uniform(-1.0, 8.0, m)
    J = rng.permutation(m)[: 3 * n // 2]
    out = np.setdiff1d(np.arange(m), J)
    AJ = A[J] * np.sqrt(sig[J])[:, None]
    H = Mq @ Mq.T + AJ.T @ AJ + beta * np.eye(n)
    kpos = {"update": k, "downdate": 0, "mixed": k // 2}[kind]
    ent = rng.choice(out, kpos, replace=False)
    lev = rng.choice(J, k - kpos, replace=False)
    W = np.hstack([(A[ent] * np.sqrt(sig[ent])[:, None]).T, (A[lev] * np.sqrt(sig[lev])[:, None]).T])
    return np.linalg.cholesky(H), W, kpos


@gpu
@pytest.mark.parametrize("beta", [1e-3, 1e-7])
@pytest.mark.parametrize("kind", ["update", "downdate", "mixed"])
def test_solver_family_against_oracle(oracle_ops, beta, kind):
    """The solver's matrices (npad 768, 32-column passes, and a 17-column one): stage checks, then the GPU's residual against
    the oracle's CHOLMOD recurrence on the same inputs."""
    rng = np.random.default_rng(int(-np.log10(beta)) * 10 + len(kind))
    for k in (32, 17):
        L, W, kpos = solver_case(rng, 768, beta, kind, k)
        Lg, info, _, st = probe_updown(L, [W], [kpos])
        what = ("solver", beta, kind, k)
        check_valid(Lg, info[0], what)
        Wh, Z, D = st
        _note("margin What", check_what(Wh, L, W, what))
        _note("margin D,Z", check_dz(Wh, Z, D, kpos, what))
        _note("margin apply", check_apply(Lg, L, W, Wh, Z, D, what))
        check_against_oracle(Lg, L, W, kpos, oracle_ops, what, "solver")


def near_singular_case(rng, n, c, kind):
    """H0 = spd with lambda_min / lambda_max = c; w of norm ~ 1.  downdate: H0 + w w' by w (leaves H0); update: H0 by w; mixed:
    H0 + w w' by (+u, -w) with a small u."""
    H0 = spd(rng, n, 1.0 / c, scale=1.0)
    w = rng.standard_normal((n, 1)) / np.sqrt(n)
    if kind == "update":
        return np.linalg.cholesky(H0), w, 1
    L = np.linalg.cholesky(H0 + w @ w.T)
    if kind == "downdate":
        return L, w, 0
    u = 1e-3 * rng.standard_normal((n, 1)) / np.sqrt(n)
    return L, np.hstack([u, w]), 1


@gpu
@pytest.mark.parametrize("c", [1e-4, 1e-8, 1e-12])
def test_near_singular_family(oracle_ops, c):
    """Valid passes that start from or end at lambda_min / ||H|| = c: whether the GPU flags the pass is recorded; a pass with
    info == 0 must have a finite factor, pass the stage checks and stay within RATIO_MAX of the oracle's residual."""
    rng = np.random.default_rng(int(-np.log10(c)))
    for kind in ("downdate", "update", "mixed"):
        L, W, kpos = near_singular_case(rng, 512, c, kind)
        Lg, info, _, st = probe_updown(L, [W], [kpos])
        what = ("near-singular", c, kind)
        print(f"[updown_gen] near-singular c={c:g} {kind}: info={int(info[0])}")
        if info[0] != 0:
            continue
        assert np.all(np.isfinite(np.tril(Lg))), what
        Wh, Z, D = st
        _note("margin What", check_what(Wh, L, W, what))
        _note("margin D,Z", check_dz(Wh, Z, D, kpos, what))
        _note("margin apply", check_apply(Lg, L, W, Wh, Z, D, what))
        check_against_oracle(Lg, L, W, kpos, oracle_ops, what, "near-singular")


def indefinite_case(rng, n, r, kpos):
    """L0 well conditioned; w = 1.5 L0[:, r] (zero above row r), so L0 L0' - w w' = L0 (I - 2.25 e_r e_r') L0' has its first
    non-positive pivot at row r; the kpos entering columns are supported below row r and leave the leading r + 1 rows alone."""
    L0 = np.linalg.cholesky(base(rng, n))
    W = np.zeros((n, kpos + 1))
    W[r + 1:, :kpos] = rng.standard_normal((n - r - 1, kpos))
    W[:, kpos] = 1.5 * L0[:, r]
    return L0, W


@gpu
@pytest.mark.parametrize("r,kpos", [(5, 0), (369, 0), (765, 0), (369, 9), (40, 31)])
def test_indefinite_downdate_is_reported_at_or_after_its_block(r, kpos):
    """A downdate that loses definiteness at row r (first block, a middle 32-row block, the last block, inside mixed passes of
    10 and 32 columns): info != 0, info - 1 a multiple of 32 and not before the block of row r."""
    rng = np.random.default_rng(r + kpos)
    L, W = indefinite_case(rng, 768, r, kpos)
    Lg, info, _, _ = probe_updown(L, [W], [kpos], stages=False)
    inf = int(info[0])
    assert inf != 0 and (inf - 1) % GB == 0 and inf - 1 >= GB * (r // GB), (r, kpos, inf)


@gpu
def test_ragged_n_identity_pad():
    """n = 300 in npad 384 as qpalm_b200_updown pads it: identity pad, zero W rows.  The leading block passes every check and
    the pad comes back exactly as the identity."""
    rng = np.random.default_rng(7)
    n, npad, k, kpos = 300, 384, 17, 9
    L0, W0 = well_case(rng, n, k, kpos)
    L = np.eye(npad)
    L[:n, :n] = L0
    W = np.zeros((npad, k))
    W[:n] = W0
    Lg, info, _, st = probe_updown(L, [W], [kpos])
    check_all(Lg, L, W, kpos, st, info[0], "ragged")
    assert np.array_equal(np.tril(Lg)[n:], np.eye(npad)[n:])
    assert not np.any(np.tril(Lg)[:n, n:])


@gpu
def test_zero_columns():
    """All of W zero: d = 1 and z = 0 exactly, so L comes back bit-identical; one zero column in a 9-column mixed pass passes
    every check."""
    rng = np.random.default_rng(8)
    L, W = well_case(rng, 512, 9, 4, zero_col=2)
    Lg, info, _, st = probe_updown(L, [W], [4])
    check_all(Lg, L, W, 4, st, info[0], "zero column")
    for k in (5, 32):
        Lg, info, _, st = probe_updown(L, [np.zeros((512, k))], [k // 2])
        assert info[0] == 0 and np.array_equal(np.tril(Lg), np.tril(L)), k
        assert np.all(st[2] == 1.0) and not np.any(st[1]), k


# ------------------------------------------------------------------------------------------------
# chains and state on one stream
# ------------------------------------------------------------------------------------------------
@gpu
def test_chain_of_passes_on_one_stream(oracle_ops):
    """100 passes at npad 1024 on one stream, alternating updates, downdates and mixed passes of 1 .. 32 columns (leaving
    columns are earlier entering ones, so every pass is valid, as in C3's sequence).  The final drift from chol(accumulated H)
    at most RATIO_MAX times the oracle chain's drift on the same passes."""
    rng = np.random.default_rng(9)
    n = 1024
    H0 = base(rng, n)
    L = np.linalg.cholesky(H0)
    pool, Ws, kp = [], [], []
    H = H0.copy()
    for p in range(100):
        kind = p % 3
        k = int(rng.integers(1, 33))
        nin = k if kind == 0 or not pool else (0 if kind == 1 else k // 2)
        nout = min(k - nin, len(pool))
        new = [rng.standard_normal(n) for _ in range(nin)]
        gone = [pool.pop(int(rng.integers(len(pool)))) for _ in range(nout)]
        pool += new
        W = np.stack(new + gone, axis=1)
        Ws.append(W)
        kp.append(nin)
        H += W[:, :nin] @ W[:, :nin].T - W[:, nin:] @ W[:, nin:].T
    Lg, info, grid, _ = probe_updown(L, Ws, kp, stages=False)
    assert not np.any(info) and np.all(np.isfinite(np.tril(Lg))), info
    Lo = L
    for W, p in zip(Ws, kp):
        Lo = oracle_pass(oracle_ops, Lo, W, p)
    Lr = np.linalg.cholesky(H)
    dg, do = np.max(np.abs(np.tril(Lg) - Lr)), np.max(np.abs(np.tril(Lo) - Lr))
    ratio = dg / max(do, gamma(n) * np.max(np.abs(Lr)))
    _note("oracle ratio chain drift", ratio)
    print(f"[updown_gen] chain drift gpu {dg:.3g} oracle {do:.3g}")
    assert ratio <= RATIO_MAX, (dg, do)


@gpu
def test_size_sequence_on_one_stream():
    """Sizes 512 -> 1024 -> 384 -> 1024 on one stream: the packet ring and Tdump are reallocated at 1024, the 384 pass runs in
    the larger buffers with packets of the earlier passes still in them, and the last pass reuses them.  The host simulates the
    sequence (each pass: chol of the leading block's L L' + W S W', the rest untouched); the final factor matches it within
    the forward error of the passes, the passes' stage outputs of the last pass pass their checks on the GPU's own input."""
    rng = np.random.default_rng(10)
    npad = 1024
    sizes, ks, kps = [512, 1024, 384, 1024], [32, 17, 9, 24], [16, 17, 0, 12]
    Ws = []
    for m, k, kp in zip(sizes, ks, kps):
        W = np.zeros((npad, k))
        W[:m, :kp] = 0.5 * rng.standard_normal((m, kp))
        W[:m, kp:] = 3e-3 * rng.standard_normal((m, k - kp))
        Ws.append(W)
    # every leading block of L L' keeps lambda_min >= lambda_min(base) ~ 1 (updates only raise it), and the leaving columns
    # of all passes together have sum ||w||^2 ~ 0.4: every downdate is valid
    Lstart = np.linalg.cholesky(base(rng, npad))
    Lg, info, grid, _ = probe_updown(Lstart, Ws, kps, sizes=sizes, stages=False)
    assert not np.any(info), info
    assert np.all(grid[:, 0] == np.minimum(np.array(sizes) // NB, grid[:, 1])), grid
    Lh = Lstart.copy()
    for m, W, kp in zip(sizes, Ws, kps):
        Wm = W[:m]
        Lh[:m, :m] = np.linalg.cholesky(Lh[:m, :m] @ Lh[:m, :m].T + Wm[:, :kp] @ Wm[:, :kp].T - Wm[:, kp:] @ Wm[:, kp:].T)
    Lg = np.tril(Lg)
    ev = np.linalg.eigvalsh(Lh @ Lh.T)
    tol = 8 * len(sizes) * (ev[-1] / ev[0]) * gamma(npad + 96) * np.max(np.abs(Lh)) * np.sqrt(npad)
    err = np.max(np.abs(Lg - Lh))
    _note("margin size sequence forward", err / tol)
    assert err <= tol, (err, tol)


# ------------------------------------------------------------------------------------------------
# grid and reproducibility
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [8, 16, 32])
def test_bit_identical_across_runs_and_grid_caps(k):
    """npad 1024 (nblk 8): the same pass twice, and with the per-group grid capped at 1 (one CTA walks every block row), 2
    and 3 (CTAs own blocks c, c + G, ...): L, What, Z and D bit-identical; the grid that ran is min(cap, nblk)."""
    rng = np.random.default_rng(20 + k)
    n = 1024
    L, W = well_case(rng, n, k, k // 2)
    ref, info, grid, st = probe_updown(L, [W], [k // 2])
    check_all(ref, L, W, k // 2, st, info[0], ("grid", k), residual=False)
    assert grid[0, 0] == min(n // NB, grid[0, 1])
    again, _, _, st2 = probe_updown(L, [W], [k // 2])
    assert np.array_equal(again, ref) and all(np.array_equal(a, b) for a, b in zip(st, st2))
    for cap in (1, 2, 3):
        Lc, info, grid, stc = probe_updown(L, [W], [k // 2], cap=cap)
        assert info[0] == 0 and grid[0, 0] == cap and grid[0, 1] == cap, (k, cap, grid)
        assert np.array_equal(Lc, ref), (k, cap)
        assert all(np.array_equal(a, b) for a, b in zip(st, stc)), (k, cap)
        print(f"[updown_gen] k={k} cap={cap}: k_fwd_multi grid {int(grid[0, 0])} x {1 if k <= 8 else 2}")


@gpu
def test_production_grid_with_several_block_rows_per_cta():
    """32-column pass at npad = 128 (gmax + 2), gmax the per-group grid limit read from the probe (the resident CTAs of
    k_fwd_multi over the two column groups): CTAs 0 and 1 own block rows c and c + gmax.  L is built directly (diagonal in
    [1, 2], strictly lower uniform(-1, 1) / n); What on the sampled block rows, D and Z on all rows, the factor formula and the
    factor formula on the sampled rows (block rows 0, 1, gmax, gmax + 1).  (The end-to-end bound needs |L||K| in full: n^3
    on the host, so it is left to the smaller cases.)"""
    import torch
    from test_gpu_dense import _mem_available
    rng = np.random.default_rng(30)
    Ls = np.tril(rng.uniform(-1, 1, (256, 256)) / 256, -1) + np.diag(rng.uniform(1, 2, 256))
    _, _, g0, _ = probe_updown(Ls, [rng.standard_normal((256, 32))], [32], stages=False)
    gmax = int(g0[0, 1])
    assert gmax > 0
    n = NB * (gmax + 2)
    need = 8 * n * n
    if torch.cuda.mem_get_info()[0] < 2 * need + (1 << 30) or _mem_available() < 4 * need:
        pytest.skip("not enough device or host memory for a %d x %d factor" % (n, n))
    Lt = rng.uniform(-1.0, 1.0, (n, n))
    Lt /= n
    for i in range(0, n, 1024):
        Lt[i:i + 1024] = np.triu(Lt[i:i + 1024], i + 1)
    Lt[np.diag_indices(n)] = rng.uniform(1.0, 2.0, n)
    L = Lt.T.copy()
    W = rng.standard_normal((n, 32))
    kpos = 20
    W[:, kpos:] *= 1e-3      # sum ||w||^2 ~ 0.12 < lambda_min(L L') ~ 1: the downdate is valid
    _, info, grid, st = probe_updown(None, [W], [kpos], Lbuf=Lt)
    Lg = Lt.T
    print(f"[updown_gen] production: npad {n}, k_fwd_multi grid {int(grid[0, 0])} x 2 (limit {int(grid[0, 1])})")
    assert info[0] == 0 and grid[0, 0] == gmax < n // NB, (info, grid)
    blocks = [0, 1, gmax, gmax + 1]
    rows = np.concatenate([np.arange(b * NB, (b + 1) * NB) for b in blocks])
    Wh, Z, D = st
    _note("margin What", check_what(Wh, L, W, "production", rows=blocks))
    _note("margin D,Z", check_dz(Wh, Z, D, kpos, "production"))
    _note("margin apply", check_apply(Lg, L, W, Wh, Z, D, "production", rows=rows))


# ------------------------------------------------------------------------------------------------
# per-panel sweep (dense.cu) and solver level
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("npad", [128, 384])
def test_per_panel_sweep(npad):
    """chol_updown (one sign per call, <= 8 columns) at npad 128 and 384: residual against the Cholesky-type bound
    8 gamma_{n+k+64} (|L_new||L_new'| + |L||L'| + |W||W'|) and forward error; at 384 it agrees with the generator form
    within the two forward-error bounds."""
    rng = np.random.default_rng(40 + npad)
    for k, kpos in ((8, 8), (5, 0), (1, 1)):
        L, W = well_case(rng, npad, k, kpos)
        Lp, info, _, _ = probe_updown(L, [W], [kpos], mode=1, stages=False)
        what = ("panel", npad, k, kpos)
        check_valid(Lp, info[0], what)
        Lp = np.tril(Lp)
        sg = signs(k, kpos)
        res = np.abs(Lp @ Lp.T - L @ L.T - (W * sg) @ W.T)
        tol = 8 * gamma(npad + k + 64) * (np.abs(Lp) @ np.abs(Lp).T + np.abs(L) @ np.abs(L).T + np.abs(W) @ np.abs(W).T)
        assert np.all(res <= tol), (what, _margin(res, tol))
        _note("margin per-panel residual", _margin(res, tol))
        _, tol_p = check_forward(Lp, L, W, kpos, what)
        if npad >= 256:
            Lg, info, _, st = probe_updown(L, [W], [kpos])
            check_all(Lg, L, W, kpos, st, info[0], what + ("gen",))
            _, tol_g = check_forward(Lg, L, W, kpos, what)
            d = np.max(np.abs(np.tril(Lg) - Lp))
            _note("margin per-panel vs generator", d / (tol_p + tol_g))
            assert d <= tol_p + tol_g, (what, d, tol_p + tol_g)


@gpu
def test_solver_passes_with_several_block_rows_per_cta():
    """A dense QP with npad > 128 gmax (the 32-column passes' grid limit, 74 on 148 SMs): forced updates
    (max_rank_update = 400, fraction 1) against refactorise-always, as test_gpu_updown.test_forced_updates_match_forced_
    refactorisations does at n = 700."""
    from test_gpu_updown import _rel, _solve
    rng = np.random.default_rng(50)
    Ls = np.tril(rng.uniform(-1, 1, (256, 256)) / 256, -1) + np.diag(rng.uniform(1, 2, 256))
    _, _, g0, _ = probe_updown(Ls, [rng.standard_normal((256, 32))], [32], stages=False)
    n = NB * (int(g0[0, 1]) + 1)
    p = problems.dense_qp(n, 1200, seed=5)
    g1, s1 = _solve("b200", p, max_rank_update=400, max_rank_update_fraction=1.0)
    g0_, s0 = _solve("b200", p, max_rank_update=0)
    print(f"[updown_gen] solver n={n}: updown_calls {s1.updown_calls} ranks {s1.updown_rank_sum} refactorizations "
          f"{s1.refactorizations} / {s0.refactorizations}")
    assert s1.updown_calls > 0 and s0.updown_calls == 0
    assert g1.status_val == g0_.status_val == 1
    assert _rel(g1.x, g0_.x) < 1e-8 and _rel(g1.y, g0_.y) < 1e-8


# ------------------------------------------------------------------------------------------------
# negative controls (no GPU)
# ------------------------------------------------------------------------------------------------
def _rejects(check, *args, **kw):
    with pytest.raises(AssertionError):
        check(*args, **kw)


def _host_pass(rng, n, k, kpos):
    """The numpy restatement's result and stage outputs for a well-conditioned pass."""
    L, W = well_case(rng, n, k, kpos)
    Wh = np.linalg.solve(L, W)
    sg = signs(k, kpos)
    M, _ = _prefix(Wh, sg)
    g = np.linalg.solve(M, Wh[:, :, None])[:, :, 0]
    D = np.sqrt(1.0 + np.sum(Wh * g, axis=1))
    Z = g / D[:, None]
    return L, W, Wh, Z, D, generator_update(L, W, kpos)


def test_checks_accept_the_host_restatement_and_reject_small_errors():
    """The float64 restatement passes every check; a relative 1e-12 change of one entry of What, of d or z, or of the updated
    factor (first block column, below the diagonal tile, in a later tile) fails the stage check that owns it -- What where L
    is diagonally dominant, z outside the last rows (both bounds are loose by the growth terms named below).  The end-to-end
    residual sums whole rows and cannot see a 1e-12 change of one entry; it and the stage checks reject one column of W with
    the wrong sign in S."""
    rng = np.random.default_rng(3)
    n, k, kpos = 384, 9, 4
    L, W, Wh, Z, D, Ln = _host_pass(rng, n, k, kpos)
    st = (Wh, Z, D)
    check_all(Ln, L, W, kpos, st, 0, "host")
    check_forward(Ln, L, W, kpos, "host")
    # the What bound carries the explicit-inverse terms |L||X||L||X| of the dense solves: a 1e-12 change stands out of it
    # where L is diagonally dominant (for this dense factor only in the first rows)
    Ld = diag_dominant_factor(rng, n)
    Whd = np.linalg.solve(Ld, W)
    check_what(Whd, Ld, W, "host, diagonally dominant")
    for i in (3, 200, 383):       # the row's largest entry
        j = int(np.argmax(np.abs(Whd[i])))
        bad = Whd.copy()
        bad[i, j] *= 1 + 1e-12
        _rejects(check_what, bad, Ld, W, ("What", i, j))
    for j in (0, 100, 383):
        bad = D.copy()
        bad[j] *= 1 + 1e-12
        _rejects(check_dz, Wh, Z, bad, kpos, ("D", j))
        if j == 383:     # z of the last rows: the Gram prefix's rounding term gamma_n |What|'|What| is above 1e-12 there
            continue
        badz = Z.copy()
        q = int(np.argmax(np.abs(Z[j])))
        badz[j, q] *= 1 + 1e-12
        _rejects(check_dz, Wh, badz, D, kpos, ("Z", j))
    # beyond the first block column the bound follows the running sums |W_r| + sum |L(r, i)||what_i|, and the off-diagonal
    # entries of this factor are far below them: there only the diagonal is seen at 1e-12 (a wrong tile start is, below)
    for i, j in ((0, 0), (100, 0), (300, 0), (300, 300), (383, 383)):
        bad = Ln.copy()
        bad[i, j] *= 1 + 1e-12
        _rejects(check_apply, bad, L, W, Wh, Z, D, ("apply", i, j))
    # the last leaving column entering instead: the pass lands on H + 2 w w'
    Lf = generator_update(L, np.hstack([W[:, :kpos], W[:, k - 1:], W[:, kpos:k - 1]]), kpos + 1)
    _rejects(check_residual, Lf, L, W, kpos, Wh, Z, D, "wrong sign")
    _rejects(check_apply, Lf, L, W, Wh, Z, D, "wrong sign")


def test_checks_reject_zero_tile_start_and_kpos_off_by_one():
    """A factor whose tiles right of the first block column start their running sums at zero (a Tdump left unwritten) fails
    the apply check and the end-to-end residual, and passes the apply check only against the zero-start reference; a mixed
    pass run with kpos one too large (a leaving column entering) or one too small (an entering column, scaled down so that
    the pass stays valid, leaving) fails the D / Z check against the intended S and the end-to-end residual."""
    rng = np.random.default_rng(4)
    n, k, kpos = 384, 17, 8
    L, W, Wh, Z, D, Ln = _host_pass(rng, n, k, kpos)
    bad = np.zeros_like(Ln)
    T = W.copy()
    for j in range(n):
        if j % NB == 0 and j > 0:
            T = W.copy()
        T -= L[:, j][:, None] * Wh[j][None, :]
        bad[:, j] = D[j] * L[:, j] + T @ Z[j]
    bad = np.tril(bad)
    check_apply(bad, L, W, Wh, Z, D, "zero start reference", tile_start_zero=True)
    _rejects(check_apply, bad, L, W, Wh, Z, D, "zero start")
    _rejects(check_residual, bad, L, W, kpos, Wh, Z, D, "zero start")
    W = W.copy()
    W[:, kpos - 1] *= 0.01
    Wh = np.linalg.solve(L, W)
    for kp in (kpos - 1, kpos + 1):
        Lw = generator_update(L, W, kp)
        Mw, _ = _prefix(Wh, signs(k, kp))
        gw = np.linalg.solve(Mw, Wh[:, :, None])[:, :, 0]
        Dw = np.sqrt(1.0 + np.sum(Wh * gw, axis=1))
        Zw = gw / Dw[:, None]
        check_apply(Lw, L, W, Wh, Zw, Dw, ("kpos", kp))
        _rejects(check_dz, Wh, Zw, Dw, kpos, ("kpos", kp))
        _rejects(check_residual, Lw, L, W, kpos, Wh, Zw, Dw, ("kpos", kp))
