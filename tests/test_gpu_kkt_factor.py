"""The signed supernodal factorization K(perm, perm) = L S L' of the KKT Newton path (csrc/sparse.cu in signed mode, driven by
csrc/kkt.cu) against float64 references, in every front kernel.

Operator entry points: `sparse_ldl` (assembly + L S L' + one solve, no refinement, on a caller's quasi-definite matrix) and
`kkt_newton` (the solver's KKT step: values, factorization, solve and iterative refinement at given inputs).

Error bounds (u = 2^-53, gamma_c = c u / (1 - c u)).  Entry (i, j) of the computed factor comes out of a_ij through: one
fused multiply-subtract per earlier column k with l_ik l_jk != 0 (fewer than N; in the 32-column tiles the products of a
block are first summed, which rounds once per term as well), one subtraction per separately accumulated block or child
update block (an extend-add; together fewer than N more), and the square root or the reciprocal-and-multiply of the
column scale (at most 3).  The classical argument for Cholesky (Higham, Accuracy and Stability, Thm 10.3), which does not
depend on the signs s_k = +-1, gives |P K P' - L S L'| <= gamma_cf |L| |L'| with cf = 2 N + 4.  The check evaluates
L S L' - P K P' in float64 itself, which adds gamma_(N+1) |L| |L'|: the factor check uses gamma_(3 N + 5).  The solves
(substitutions with the same column scales, Thm 10.4) add two more triangular solves: (K + dK) x = b with
|dK| <= gamma_(3 cf) |L| |L'|, so |b - K x| <= gamma_(3 cf) |L| |L'| |x| + gamma_(N+1) (|K| |x| + |b|), the last term for
the float64 residual.

Exact sign algebra: fstep_signed with s = +1 performs exactly the operations of fstep, and every kernel multiplies by the
sign (+-1.0, exact) where the positive-definite mode multiplies by 1.0; with s = -1 everywhere every operation is the
negated one of the positive-definite factorization of -K.  Hence n_pos = N must reproduce the positive-definite factor and
solution bit for bit, and n_pos = 0 the factor of -K bit for bit and the negated solution.
"""
import ctypes as C
import json
import os
from contextlib import contextmanager

import numpy as np
import pytest
import scipy.sparse as sp

from qpalm_b200 import abi, problems
from qpalm_b200.interface import load_library
from qpalm_b200.sparse import kkt_newton, sparse_ldl, sparse_newton, symbolic

U = 2.0 ** -53
SMALL_MAX_NF = 160   # kSmallMaxNf of csrc/sparse.cu: larger fronts go to k_mf_front or to the per-block launches


def gamma(c):
    return c * U / (1.0 - c * U)


@contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)


def launched(fn):
    """Runs fn() with every launch of the library timed and returns (fn(), {kernel name: launches})."""
    lib = load_library("b200")
    lib.qpalm_b200_prof_enable.argtypes = [C.c_char_p]
    lib.qpalm_b200_prof_report.argtypes = [C.c_char_p, C.c_size_t]
    lib.qpalm_b200_prof_enable(b"*")
    try:
        out = fn()
    finally:
        buf = C.create_string_buffer(1 << 20)   # one call: a report also clears the log
        lib.qpalm_b200_prof_report(buf, len(buf))
        lib.qpalm_b200_prof_enable(b"")
    return out, {k: v["launches"] for k, v in json.loads(buf.value.decode()).items()}


# ---------------------------------------------------------------------------------------------------------------------
# matrix families (all quasi-definite: K = [[P, B'], [B, -C]] up to a symmetric permutation, P and C positive definite;
# original columns < n_pos are the positive ones)
# ---------------------------------------------------------------------------------------------------------------------
def _spd(k, rng, cond):
    if k == 0:
        return np.zeros((0, 0))
    Qm, _ = np.linalg.qr(rng.standard_normal((k, k)))
    return (Qm * np.logspace(0.0, -np.log10(cond), k)) @ Qm.T


def qd_dense(N, n_pos, seed, cond_P=10.0, c_min=1.0):
    """Dense quasi-definite matrix: one root front (nr = 0).  P has condition cond_P, C eigenvalues in [c_min, 1]."""
    rng = np.random.default_rng(seed)
    K = np.zeros((N, N))
    K[:n_pos, :n_pos] = _spd(n_pos, rng, cond_P)
    K[n_pos:, n_pos:] = -_spd(N - n_pos, rng, 1.0 / c_min)
    B = 0.5 * rng.standard_normal((N - n_pos, n_pos))
    K[n_pos:, :n_pos] = B
    K[:n_pos, n_pos:] = B.T
    return 0.5 * (K + K.T)


def _relabel_positives_first(K, pos):
    order = np.concatenate([np.flatnonzero(pos), np.flatnonzero(~pos)])
    return K[np.ix_(order, order)], int(pos.sum())


def qd_bordered(tree, seed, frac_pos=0.6, scale_P=1.0, c_min=1.0):
    """Bordered block-diagonal pattern given by `tree`: a leaf is the size of an independent dense block, a node
    (s, [children]) a separator of size s coupled densely to every variable of its subtree (nested dissection shape).
    Signs are drawn per variable; P and C are diagonally dominant, then rows / columns of positive variables are scaled by a
    logspace(0, -log10(scale_P) / 2) diagonal (condition of P about scale_P) and C by c_min."""
    rng = np.random.default_rng(seed)

    def build(t):
        if isinstance(t, int):
            return np.ones((t, t), dtype=bool)
        s, children = t
        kids = [build(c) for c in children]
        n = sum(k.shape[0] for k in kids) + s
        M = np.zeros((n, n), dtype=bool)
        o = 0
        for k in kids:
            M[o:o + k.shape[0], o:o + k.shape[0]] = k
            o += k.shape[0]
        M[o:, :] = True
        M[:, o:] = True
        return M

    pat = build(tree)
    N = pat.shape[0]
    pos = rng.random(N) < frac_pos
    M = np.where(pat, rng.standard_normal((N, N)), 0.0)
    M = np.triu(M, 1)
    M = M + M.T
    same = pos[:, None] == pos[None, :]
    dom = np.sum(np.abs(np.where(same, M, 0.0)), axis=1) + 1.0
    K = M.copy()
    K[np.diag_indices(N)] = np.where(pos, dom, -dom)
    dsc = np.ones(N)
    dsc[pos] = np.logspace(0.0, -0.5 * np.log10(scale_P), int(pos.sum()))
    dsc[~pos] = np.sqrt(c_min)
    K = dsc[:, None] * K * dsc[None, :]
    Kp, n_pos = _relabel_positives_first(K, pos)
    patp, _ = _relabel_positives_first(pat.astype(float), pos)
    return Kp, n_pos, patp != 0


def lower_csc(K, pattern=None):
    """Lower triangle of K in CSC with every entry of `pattern` stored (explicit zeros stay), rows ascending."""
    pat = np.ones_like(K, dtype=bool) if pattern is None else (pattern | (K != 0))
    pat = np.tril(pat | np.eye(K.shape[0], dtype=bool))
    N = K.shape[0]
    p = np.zeros(N + 1, dtype=np.int64)
    rows, vals = [], []
    for j in range(N):
        r = np.flatnonzero(pat[:, j])
        rows.append(r)
        vals.append(K[r, j])
        p[j + 1] = p[j] + r.size
    return abi.CSC(N, N, p, np.concatenate(rows), np.concatenate(vals), -1)


def kkt_csc(p, sigma, active, beta):
    """The KKT matrix exactly as kkt_create / k_kkt_values build it: columns j < n hold [j if Q stores no diagonal] + the
    stored lower entries of Q + the rows n + i of A; column n + i holds the diagonal.  Inactive rows keep their (zero)
    entries and a -1 diagonal.  Returns (lower CSC, dense K, n_pos = n)."""
    n, m = p.n, p.m
    Qp, Qi, Qx = p.Q.p, p.Q.i, p.Q.x
    Ap, Ai, Ax = p.A.p, p.A.i, p.A.x
    colp, rows, vals = [0], [], []
    for j in range(n):
        qr, qv = Qi[Qp[j]:Qp[j + 1]], Qx[Qp[j]:Qp[j + 1]]
        keep = qr >= j
        qr, qv = qr[keep], qv[keep]
        has_diag = bool((qr == j).any())
        if not has_diag:
            rows.append([j]); vals.append([beta])
        rows.append(qr); vals.append(np.where(qr == j, qv + beta, qv + 0.0))
        ar, av = Ai[Ap[j]:Ap[j + 1]], Ax[Ap[j]:Ap[j + 1]]
        rows.append(n + ar); vals.append(np.where(active[ar] != 0, av, 0.0))
        colp.append(colp[-1] + (0 if has_diag else 1) + qr.size + ar.size)
    for i in range(m):
        rows.append([n + i]); vals.append([-1.0 / sigma[i] if active[i] else -1.0])
        colp.append(colp[-1] + 1)
    r = np.concatenate([np.asarray(x, dtype=np.int64) for x in rows])
    v = np.concatenate([np.asarray(x, dtype=np.float64) for x in vals])
    Kc = abi.CSC(n + m, n + m, np.asarray(colp, dtype=np.int64), r, v, -1)
    Kl = sp.csc_matrix((v, r, np.asarray(colp)), shape=(n + m, n + m)).toarray()
    return Kc, Kl + np.tril(Kl, -1).T, n


def signs_permuted(perm, n_pos):
    return np.where(np.asarray(perm) >= n_pos, -1.0, 1.0)


# ---------------------------------------------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------------------------------------------
def check_factor_and_solve(K, n_pos, L, perm, x, b):
    N = K.shape[0]
    s = signs_permuted(perm, n_pos)
    Kp = K[np.ix_(perm, perm)]
    absLL = np.abs(L) @ np.abs(L).T
    R = (L * s) @ L.T - Kp
    cf = 2 * N + 4
    bad = np.abs(R) > gamma(3 * N + 5) * absLL
    assert not bad.any(), f"factor: {bad.sum()} entries above the bound, worst ratio {np.max(np.abs(R)[bad] / np.maximum(absLL[bad], 1e-300)):.3g}"
    assert np.all(np.triu(L, 1) == 0.0)
    assert np.all(np.diag(L) > 0.0)
    # solve: componentwise backward error
    assert np.all(np.isfinite(x))
    xp = x[perm]
    r = (b - K @ x)[perm]
    bound = gamma(3 * cf) * (absLL @ np.abs(xp)) + gamma(N + 1) * (np.abs(Kp) @ np.abs(xp) + np.abs(b[perm]))
    over = np.abs(r) > bound
    assert not over.any(), f"solve: {over.sum()} residual entries above the bound, worst ratio {np.max(np.abs(r)[over] / bound[over]):.3g}"
    # forward error against LAPACK: condition number times the backward error, which is relative to |L| |L'| (the growth
    # of the factor over K enters)
    xr = np.linalg.solve(K, b)
    kappa = np.linalg.norm(K, 1) * np.linalg.norm(np.linalg.inv(K), 1)
    growth = max(1.0, np.max(absLL) / np.max(np.abs(K)))
    assert np.max(np.abs(x - xr)) <= 20 * N * U * kappa * growth * max(np.max(np.abs(xr)), 1e-300)


def run_ldl(K, n_pos, b, pattern=None, **kw):
    Kc = lower_csc(K, pattern)
    rc, x, L, perm, panels = sparse_ldl(Kc, n_pos, b, **kw)
    return rc, x, L, perm, panels, Kc


# ---------------------------------------------------------------------------------------------------------------------
# 1. dense quasi-definite matrices: one root front, both sides of kSmallMaxNf, every split of the signs
# ---------------------------------------------------------------------------------------------------------------------
DENSE_N = [1, 2, 31, 32, 33, 160, 161, 200, 257]
DENSE_CASES = sorted({(N, q) for N in DENSE_N for q in (0, 1, N // 2, N - 1, N)})


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_pos", DENSE_CASES, ids=[f"N{N}-pos{q}" for N, q in DENSE_CASES])
def test_dense_quasi_definite_factor_and_solve(N, n_pos):
    K = qd_dense(N, n_pos, seed=1000 * N + n_pos)
    b = np.random.default_rng(N + 7 * n_pos).standard_normal(N)
    sym = symbolic(lower_csc(K), None)
    assert sym["nsuper"] == 1 and sym["max_nf"] == N and sym["max_ns"] == N   # one root front, nr = 0
    rc, x, L, perm, _, _ = run_ldl(K, n_pos, b, want_factor=True)
    assert rc == 0
    assert np.array_equal(perm, sym["perm"])
    check_factor_and_solve(K, n_pos, L, perm, x, b)


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_pos", [(33, 16), (161, 80), (257, 129)], ids=["N33", "N161", "N257"])
@pytest.mark.parametrize("cond_P,c_min", [(1e8, 1e-8), (1e1, 1e-8), (1e8, 1.0)], ids=["P1e8-C1e-8", "P1e1-C1e-8", "P1e8-C1"])
def test_dense_ill_conditioned_blocks(N, n_pos, cond_P, c_min):
    """P with condition 1e8 and / or C down to 1e-8 (sigma up to 1e8): the bounds are relative to |L| |L'| and hold as well."""
    K = qd_dense(N, n_pos, seed=N + int(np.log10(cond_P)), cond_P=cond_P, c_min=c_min)
    b = np.random.default_rng(N).standard_normal(N)
    rc, x, L, perm, _, _ = run_ldl(K, n_pos, b, want_factor=True)
    assert rc == 0
    check_factor_and_solve(K, n_pos, L, perm, x, b)


# ---------------------------------------------------------------------------------------------------------------------
# 2. bordered block-diagonal matrices: extend-add into large fronts, nr > 0, several levels
# ---------------------------------------------------------------------------------------------------------------------
BORDERED = {
    # name: (tree, scale_P, c_min); fronts (ns, nr) by level as the analysis builds them (the ordering merges one block
    # into each separator)
    "all_small": ((40, [100, 100, 100]), 1.0, 1.0),                 # (100, 40) x 2 | (140, 0): k_mf_small only
    "small_children_large_root": ((60, [50, 50, 150]), 1.0, 1.0),   # (50, 60) x 2 | (210, 0)
    "mixed_level": ((40, [150, 150, 20]), 1.0, 1.0),                # (20, 40), (150, 40) | (190, 0)
    "large_children_large_root": ((170, [100, 100, 100]), 1.0, 1.0),  # (100, 170) x 2 | (270, 0)
    "nested": ((50, [(60, [40, 40, 120]), (30, [130, 20])]), 1.0, 1.0),   # 3 small | (160, 50) | (230, 0)
    "nested_ill": ((40, [(100, [30, 30, 30]), (60, [120, 20])]), 1e8, 1e-8),   # P condition ~1e8, C ~1e-8
}


def _bordered(name, **kw):
    tree, scale_P, c_min = BORDERED[name]
    args = dict(seed=1, scale_P=scale_P, c_min=c_min)
    args.update(kw)
    return qd_bordered(tree, **args)


def front_shapes(sym):
    ns = np.diff(sym["sn_first"])
    nr = np.diff(sym["rows_off"])
    return ns, nr, ns + nr


def test_bordered_families_have_the_intended_fronts():
    """Host-only: the symbolic analysis (the same one sparse_ldl runs) gives the front shapes each case is meant to reach:
    extend-add into fronts on both sides of kSmallMaxNf, large fronts with nr > 0, levels that mix small and large fronts."""
    sym = {}
    for name in BORDERED:
        K, n_pos, pat = _bordered(name)
        sym[name] = symbolic(lower_csc(K, pat), None)
    big_nr = lambda name: bool(((front_shapes(sym[name])[2] > SMALL_MAX_NF) & (front_shapes(sym[name])[1] > 0)).any())
    assert front_shapes(sym["all_small"])[2].max() <= SMALL_MAX_NF and sym["all_small"]["nlevels"] == 2
    ns, nr, nf = front_shapes(sym["small_children_large_root"])
    assert nf[:-1].max() <= SMALL_MAX_NF < nf[-1] and nr[-1] == 0
    for name in ("mixed_level", "large_children_large_root", "nested", "nested_ill"):
        assert big_nr(name), name
    ns, nr, nf = front_shapes(sym["mixed_level"])
    lvl0 = sym["mixed_level"]["lvl_sn"][:sym["mixed_level"]["lvl_ptr"][1]]
    assert nf[lvl0].min() <= SMALL_MAX_NF < nf[lvl0].max()     # small fronts in a level of large ones
    for name in ("nested", "nested_ill"):
        assert sym[name]["nlevels"] >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BORDERED))
def test_bordered_quasi_definite_factor_and_solve(name):
    K, n_pos, pat = _bordered(name)
    N = K.shape[0]
    b = np.random.default_rng(3).standard_normal(N)
    rc, x, L, perm, _, _ = run_ldl(K, n_pos, b, pattern=pat, want_factor=True)
    assert rc == 0
    check_factor_and_solve(K, n_pos, L, perm, x, b)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the solver's own KKT patterns
# ---------------------------------------------------------------------------------------------------------------------
SOLVER_KKT = {
    "grid24": lambda: problems.grid_qp(24, seed=2),
    "rand_300_600": lambda: problems.random_qp(300, 600, 0.02, 0.01, seed=3),
    "rand_700_900": lambda: problems.random_qp(700, 900, 0.2, 0.1, seed=5),
}
# (max front rows, fronts above kSmallMaxNf) of their KKT patterns: grid24 stays in k_mf_small, the random ones reach the
# large-front kernels
SOLVER_KKT_FRONTS = {"grid24": (51, 0), "rand_300_600": (263, 6), "rand_700_900": (701, 33)}


def _solver_kkt(name, sigma_max=20.0):
    p = SOLVER_KKT[name]()
    rng = np.random.default_rng(len(name))
    sigma = 0.5 + (sigma_max - 0.5) * rng.random(p.m)
    act = (rng.random(p.m) < 0.5).astype(np.int64)
    Kc, K, n_pos = kkt_csc(p, sigma, act, 1e-3)
    return Kc, K, n_pos


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SOLVER_KKT))
@pytest.mark.parametrize("sigma_max", [20.0, 1e8], ids=["sigma20", "sigma1e8"])
def test_solver_kkt_patterns_factor_and_solve(name, sigma_max):
    Kc, K, n_pos = _solver_kkt(name, sigma_max)
    sym = symbolic(Kc, None)
    assert (sym["max_nf"], int((front_shapes(sym)[2] > SMALL_MAX_NF).sum())) == SOLVER_KKT_FRONTS[name]
    b = np.random.default_rng(9).standard_normal(K.shape[0])
    rc, x, L, perm, _ = sparse_ldl(Kc, n_pos, b, want_factor=True)
    assert rc == 0
    check_factor_and_solve(K, n_pos, L, perm, x, b)


# ---------------------------------------------------------------------------------------------------------------------
# coverage: every signed-mode kernel is launched, with mixed-sign, ragged and nr > 0 large fronts
# ---------------------------------------------------------------------------------------------------------------------
def _blocks(sym, n_pos):
    """(nf, w, mixed) for every 32-column diagonal block of every front."""
    s = signs_permuted(sym["perm"], n_pos)
    out = []
    for f0, f1, r0, r1 in zip(sym["sn_first"][:-1], sym["sn_first"][1:], sym["rows_off"][:-1], sym["rows_off"][1:]):
        for k0 in range(f0, f1, 32):
            blk = s[k0:min(k0 + 32, f1)]
            out.append((f1 - f0 + r1 - r0, blk.size, bool((blk > 0).any() and (blk < 0).any())))
    return out


@pytest.mark.gpu
def test_signed_kernels_are_all_reached():
    big = qd_dense(161, 80, seed=5)
    Kb, qb, patb = _bordered("nested")
    small = qd_dense(33, 16, seed=6)
    b161, bb, b33 = np.ones(161), np.ones(Kb.shape[0]), np.ones(33)
    blocks = _blocks(symbolic(lower_csc(big), None), 80) + _blocks(symbolic(lower_csc(Kb, patb), None), qb)
    assert any(nf > SMALL_MAX_NF and mixed for nf, w, mixed in blocks), "no mixed-sign diagonal block in a large front"
    assert any(nf > SMALL_MAX_NF and w < 32 for nf, w, mixed in blocks), "no ragged diagonal block in a large front"
    ns, nr, nf = front_shapes(symbolic(lower_csc(Kb, patb), None))
    assert ((nf > SMALL_MAX_NF) & (nr > 0)).any()

    (rc, *_), k = launched(lambda: run_ldl(small, 16, b33))
    assert rc == 0 and k.get("k_mf_small", 0) > 0 and k.get("k_sp_apply_sign", 0) == 1
    for K, q, pat, b in ((big, 80, None, b161), (Kb, qb, patb, bb)):
        (rc, *_), k = launched(lambda: run_ldl(K, q, b, pattern=pat))
        assert rc == 0
        for name in ("k_mf_front", "k_mf_fwd_big", "k_mf_bwd_big", "k_sp_apply_sign"):
            assert k.get(name, 0) > 0, (name, k)
        with env(QPALM_B200_MF_PER_BLOCK=1):
            (rc, *_), k = launched(lambda: run_ldl(K, q, b, pattern=pat))
        assert rc == 0 and k.get("k_mf_front", 0) == 0
        for name in ("k_mf_extend", "k_mf_diag", "k_mf_trsm", "k_mf_syrk"):
            assert k.get(name, 0) > 0, (name, k)


# ---------------------------------------------------------------------------------------------------------------------
# 4. exact sign algebra: all +1 is the positive-definite mode, all -1 the positive-definite mode of -K
# ---------------------------------------------------------------------------------------------------------------------
def _pd_newton(Kpd, b, pattern=None):
    """Positive-definite factor and solution of Kpd through the Schur path's operator (one inactive single-entry row)."""
    N = Kpd.shape[0]
    A = abi.CSC(1, N, np.concatenate([[0], np.ones(N, dtype=np.int64)]), np.zeros(1, dtype=np.int64), np.ones(1))
    d, L, perm, _ = sparse_newton(lower_csc(Kpd, pattern), A, np.ones(1), np.zeros(1, dtype=np.int64), 0.0, b, want_factor=True)
    return d, L, perm


SIGN_CASES = [("dense", 31), ("dense", 33), ("dense", 161), ("dense", 257),
              ("bordered", "mixed_level"), ("bordered", "nested"), ("bordered", "large_children_large_root")]


def _sign_case(kind, arg, sign):
    if kind == "dense":
        N = arg
        K = qd_dense(N, N if sign > 0 else 0, seed=N)
        return K, None
    K, n_pos, pat = _bordered(arg, seed=11, frac_pos=1.0 if sign > 0 else 0.0)
    return K, pat


@pytest.mark.gpu
@pytest.mark.parametrize("kind,arg", SIGN_CASES, ids=[f"{k}-{a}" for k, a in SIGN_CASES])
@pytest.mark.parametrize("sign", [+1, -1], ids=["all_plus", "all_minus"])
def test_uniform_signs_are_bit_identical_to_the_positive_definite_mode(kind, arg, sign):
    K, pat = _sign_case(kind, arg, sign)
    N = K.shape[0]
    b = np.random.default_rng(N).standard_normal(N)
    rc, x, L, perm, _, _ = run_ldl(K, N if sign > 0 else 0, b, pattern=pat, want_factor=True)
    assert rc == 0
    d, Lpd, perm_pd = _pd_newton(sign * K, b, pat)
    assert np.array_equal(perm, perm_pd), "the two analyses ordered differently"
    assert np.array_equal(L, Lpd)
    assert np.array_equal(x, sign * d)


# ---------------------------------------------------------------------------------------------------------------------
# 5. path equivalence in signed mode: per-block launches, every cluster size, generic solves, repeated runs
# ---------------------------------------------------------------------------------------------------------------------
CONFIGS = [("per_block", dict(QPALM_B200_MF_PER_BLOCK=1)),
           ("cluster1", dict(QPALM_B200_MF_PER_BLOCK=0, QPALM_B200_MF_CLUSTER=1)),
           ("cluster2", dict(QPALM_B200_MF_PER_BLOCK=0, QPALM_B200_MF_CLUSTER=2)),
           ("cluster8", dict(QPALM_B200_MF_PER_BLOCK=0, QPALM_B200_MF_CLUSTER=8)),
           ("cluster16", dict(QPALM_B200_MF_PER_BLOCK=0, QPALM_B200_MF_CLUSTER=16)),
           ("generic_solves", dict(QPALM_B200_MF_FWD_GENERIC=1)),
           ("default", {}), ("default_again", {})]
PATH_CASES = ["dense257", "large_children_large_root", "nested", "mixed_level", "rand_300_600", "rand_700_900"]


def _path_case(name):
    if name == "dense257":
        return lower_csc(qd_dense(257, 100, seed=4)), 100
    if name in BORDERED:
        K, n_pos, pat = _bordered(name)
        return lower_csc(K, pat), n_pos
    Kc, _, n_pos = _solver_kkt(name)
    return Kc, n_pos


@pytest.mark.gpu
@pytest.mark.parametrize("name", PATH_CASES)
def test_signed_paths_are_bit_identical(name):
    Kc, n_pos = _path_case(name)
    nnzL = symbolic(Kc, None)["nnzL"]
    b = np.random.default_rng(2).standard_normal(Kc.ncol)
    out = {}
    for cfg, e in CONFIGS:
        with env(**e):
            rc, x, _, _, panels = sparse_ldl(Kc, n_pos, b, panels_len=nnzL)
        assert rc == 0, cfg
        out[cfg] = (x, panels)
    x0, p0 = out["per_block"]
    for cfg, (x, panels) in out.items():
        assert np.array_equal(panels, p0), cfg
        assert np.array_equal(x, x0), cfg


# ---------------------------------------------------------------------------------------------------------------------
# 6. failure reporting: a matrix that is not quasi-definite returns >= 1000, never a silent NaN
# ---------------------------------------------------------------------------------------------------------------------
def _with_extra_column(K, n_pos, pattern, where, value, coupled):
    """K with one extra column carrying `value` on its diagonal and zeros elsewhere: a negative one (original index N,
    after the negatives) or a positive one (original index n_pos, before the negatives).  coupled: its zeros are stored
    (the column joins the fronts of its neighbours, as an inactive KKT row does); otherwise it is a front of its own."""
    N = K.shape[0]
    at = N if where == "neg" else n_pos
    K2 = np.insert(np.insert(K, at, 0.0, axis=0), at, 0.0, axis=1)
    K2[at, at] = value
    pat = np.ones_like(K, dtype=bool) if pattern is None else pattern
    pat = np.insert(np.insert(pat, at, coupled, axis=0), at, coupled, axis=1)
    pat[at, at] = True
    return K2, n_pos + (1 if where == "pos" else 0), pat, at


@pytest.mark.gpu
@pytest.mark.parametrize("base", ["dense33", "dense200", "nested"])
@pytest.mark.parametrize("where,bad,good", [("neg", 0.5, -0.5), ("pos", 0.0, 2.0)], ids=["positive_in_C", "zero_in_P"])
@pytest.mark.parametrize("coupled", [False, True], ids=["decoupled", "stored_zeros"])
def test_not_quasi_definite_is_reported(base, where, bad, good, coupled):
    """A pivot of the wrong sign must give rc >= 1000, not a silent NaN.  A decoupled column is a front of its own, so the
    flag names it exactly; a column that shares a front (the root front in these cases) flags a pivot of that front: the NaN it
    leaves spreads to the later pivots, which flag as well."""
    if base.startswith("dense"):
        N = int(base[5:])
        K, n_pos, pat = qd_dense(N, N // 2, seed=N), N // 2, None
    else:
        K, n_pos, pat = _bordered(base)
    rhs_rng = np.random.default_rng(1)
    for value, healthy in ((good, True), (bad, False)):
        K2, q2, pat2, at = _with_extra_column(K, n_pos, pat, where, value, coupled)
        b = rhs_rng.standard_normal(K2.shape[0])
        rc, x, L, perm, _, _ = run_ldl(K2, q2, b, pattern=pat2, want_factor=True)
        if healthy:
            assert rc == 0
            check_factor_and_solve(K2, q2, L, perm, x, b)
            continue
        assert rc >= 1000
        sym = symbolic(lower_csc(K2, pat2), None)
        flagged = rc - 1001
        s_bad = sym["sn_of_col"][np.flatnonzero(perm == at)[0]]
        if coupled:
            assert sym["sn_of_col"][flagged] == s_bad, "the flag is outside the front of the broken column"
        else:
            assert perm[flagged] == at, "the flagged pivot is not the broken column"


# ---------------------------------------------------------------------------------------------------------------------
# 7. the KKT step (kkt_newton): values, factorization, solve and iterative refinement at given inputs
# ---------------------------------------------------------------------------------------------------------------------
class _P:   # minimal problem record for kkt_csc
    def __init__(self, Q, A):
        self.Q, self.A, self.n, self.m = Q, A, Q.ncol, A.nrow


def _step_case(name, seed=0):
    """(Q lower CSC, A CSC, sigma, active, beta) of the named KKT-step case."""
    rng = np.random.default_rng(seed)
    n, m = 60, 45
    A = sp.random(m, n, density=0.06, format="lil", random_state=rng, data_rvs=lambda k: 0.3 * rng.standard_normal(k))
    M = sp.random(n, n, density=0.02, format="csc", random_state=rng, data_rvs=rng.standard_normal)
    Qd = (M @ M.T).toarray() + np.diag(0.5 + rng.random(n))
    sigma = 0.5 + 19.5 * rng.random(m)
    act = (rng.random(m) < 0.6).astype(np.int64)
    beta = 1e-2
    drop_diag = np.zeros(n, dtype=bool)
    if name in ("empty_A_columns", "all_inactive"):
        A[:, :15] = 0.0                                   # A columns with no entries
    if name == "empty_rows":
        A[:10, :] = 0.0                                   # rows with no entries, active ones included
        act[:10] = 1
    if name == "all_inactive":
        act[:] = 0
    if name == "q_without_diagonal":
        beta = 1.0                                        # the only curvature of a variable Q and A leave empty
        drop_diag[rng.choice(n, 12, replace=False)] = True   # Q stores no diagonal (and no column) there: the structural beta
        Qd[drop_diag, :] = 0.0
        Qd[:, drop_diag] = 0.0
    if name == "beta_zero":
        beta = 0.0
    if name == "sigma_1e8":
        sigma = np.logspace(-1, 8, m)
        rng.shuffle(sigma)
    A = sp.csc_matrix(A)
    A.eliminate_zeros()
    Ql = sp.csc_matrix(np.tril(Qd))
    Ql.eliminate_zeros()
    if name == "q_without_diagonal":
        assert all(j not in Ql.indices[Ql.indptr[j]:Ql.indptr[j + 1]] for j in np.flatnonzero(drop_diag))
    return abi.CSC.from_scipy(Ql, stype=-1), abi.CSC.from_scipy(A), sigma, act, beta


STEP_CASES = ["basic", "empty_A_columns", "empty_rows", "all_inactive", "q_without_diagonal", "beta_zero", "sigma_1e8"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", STEP_CASES)
def test_kkt_newton_step(name):
    """d = (Q + A_J' Sigma_J A_J + beta I)^{-1} rhs.  Refinement: after the first solve |K z - r| is bounded a priori by
    gamma_(3 cf) |L| |L'| |z| (module docstring).  This bound is evaluated below with the factor of the same K (sparse_ldl
    on the matrix built as kkt_create builds it; its values are the same doubles, so the analysis and the factor are the
    same); on the well-scaled cases (sigma in [0.5, 20]) it must lie two orders of magnitude below the refinement threshold
    1e-10 max(|K z|, |r|), so no correction may be applied and d must be the first solve bit for bit."""
    Q, A, sigma, act, beta = _step_case(name)
    n, m = Q.ncol, A.nrow
    rhs = np.random.default_rng(4).standard_normal(n)
    rc, d, refine, (res, ref) = kkt_newton(Q, A, sigma, act, beta, rhs)
    assert rc == 0
    Qf = Q.to_scipy().toarray()
    Ad = A.to_scipy().toarray()
    J = act != 0
    H = Qf + Ad[J].T @ (sigma[J, None] * Ad[J]) + beta * np.eye(n)
    dref = np.linalg.solve(H, rhs)
    Kc, K, n_pos = kkt_csc(_P(Q, A), sigma, act, beta)
    N = n + m
    kappa = np.linalg.norm(K, 1) * np.linalg.norm(np.linalg.inv(K), 1)
    assert np.max(np.abs(d - dref)) <= 20 * N * U * kappa * max(np.max(np.abs(dref)), 1e-300)
    r_full = np.concatenate([rhs, np.zeros(m)])
    rc2, z, L, perm, _ = sparse_ldl(Kc, n_pos, r_full, want_factor=True)
    assert rc2 == 0
    check_factor_and_solve(K, n_pos, L, perm, z, r_full)
    if name == "sigma_1e8":
        assert refine <= 3
        assert res <= max(1e-10 * ref, 1e-12)
        return
    zp = np.abs(z[perm])
    predicted = np.max(gamma(3 * (2 * N + 4)) * ((np.abs(L) @ (np.abs(L).T @ zp))) + gamma(N + 1) * (np.abs(K[np.ix_(perm, perm)]) @ zp))
    threshold = max(1e-10 * max(np.max(np.abs(K @ z)), np.max(np.abs(r_full))), 1e-12)
    assert predicted <= 1e-2 * threshold, (predicted, threshold)
    assert refine == 0, f"{refine} refinement corrections on a well-scaled step (residual {res:.3g}, threshold {threshold:.3g})"
    assert np.array_equal(d, z[:n])
