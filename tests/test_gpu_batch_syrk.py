"""The persistent batch engine's tile-stationary SYRK (batchp.cu cta_syrk) against float64, in both CTA shapes.

H = base + A_P' diag(w^2) A_P - A_N' diag(w^2) A_N, with base the instance's H0 updated in place (the incremental H record)
or sscale * Q from the shared matrix (the rebuild from c Q), for list lengths across the stage boundaries of both shapes
(24 and 36 entries) and the group boundaries of the n x n triangle, up to the benchmark's m = 949.  The factor of every
result is checked as in test_gpu_batch_cta."""
import numpy as np
import pytest

from test_gpu_batch_cta import EPS, check_factor, gram, probe_newton, spd, sym

pytestmark = pytest.mark.gpu

M_BENCH = 949
LENGTHS = ((0, 0), (1, 0), (0, 1), (23, 1), (24, 0), (25, 12), (35, 1), (36, 0), (37, 36), (71, 2), (72, 0),
           (73, 60), (300, 40), (500, 449), (949, 0))


def _cases(rng, A, n, from_q):
    m = A.shape[0]
    insts, refs = [], []
    for kp, kn in LENGTHS:
        rows = rng.permutation(m)
        pr, nr = rows[:kp], rows[kp:kp + kn]
        pw, nw = 10 ** rng.uniform(-2, 1, kp), 10 ** rng.uniform(-2, 1, kn)
        it = dict(pos=(pr, pw), neg=(nr, nw), rhs=rng.standard_normal(n))
        if not from_q:
            it["H0"] = spd(rng, n, 10.0) + gram(A, nr, nw)   # the leaving rows are part of H0: H stays positive definite
        insts.append(it)
        refs.append((pr, pw, nr, nw))
    return insts, refs


@pytest.mark.parametrize("shape", (3, 4), ids=["shape3", "shape4"])
@pytest.mark.parametrize("n", [45, 128, 183, 240])
@pytest.mark.parametrize("from_q", [False, True], ids=["in_place", "from_q"])
def test_syrk_stream(shape, n, from_q):
    rng = np.random.default_rng(1000 + n + 7 * from_q)
    A = rng.standard_normal((M_BENCH, n)) / np.sqrt(n)
    sscale = 0.37
    Q = None
    if from_q:
        # every instance's minus rows are in the shared base, so that H stays positive definite
        Q = spd(rng, n, 10.0) + gram(A, np.arange(M_BENCH), np.full(M_BENCH, 10.0)) / sscale
    insts, refs = _cases(rng, A, n, from_q)
    H, L, dfu, daf, info = probe_newton(shape, A, insts, from_q=Q, sscale=sscale)
    for b, (pr, pw, nr, nw) in enumerate(refs):
        H0 = sscale * Q if from_q else insts[b]["H0"]
        ref = H0 + gram(A, pr, pw) - gram(A, nr, nw)
        # K = |P| + |N| products of w^2 a_i a_j added to the base: gamma_{K+3} T entrywise with T = |base| + sum w^2 |a_i a_j|;
        # the float64 reference adds gamma_{K+1} T; 2 (K + 4) eps covers both (the bound of test_syrk_lists)
        T = np.abs(H0) + gram(np.abs(A), pr, pw) + gram(np.abs(A), nr, nw)
        tol = 2 * (len(pr) + len(nr) + 4) * EPS * T
        err = np.abs(np.tril(H[b]) - np.tril(ref))
        what = (shape, n, from_q, len(pr), len(nr))
        assert np.all(err <= np.tril(tol)), (what, float(np.max(err - tol)))
        if len(pr) + len(nr) == 0 and not from_q:
            assert np.array_equal(H[b], np.tril(H0)), what
        assert info[b] == 0, what
        check_factor(L[b], sym(H[b]), what)
