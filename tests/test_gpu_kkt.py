"""SURVEY.md 8 row f3 -- the KKT factorization path of the Newton step (kkt.cu).

Reference: FACTORIZE_KKT branch of newton_set_direction (src/newton.c:22-95), qpalm_form_kkt / kkt_solve
(src/solver_interface.c:119-247), selection criterion src/solver_interface.c:20-66 (LADEL build).  The KKT system and the
Schur complement give the SAME Newton direction, so the trajectory must agree with the reference's Schur path (CHOLMOD
build, oracle/_ref) and with the oracle to the north-star gates: same status, x / y 1e-8, iteration counts within 5 %."""
import ctypes

import numpy as np
import pytest

from conftest import HAS_REF
from qpalm_b200 import problems
from qpalm_b200.interface import Qpalm

pytestmark = pytest.mark.gpu
libc = ctypes.CDLL("libc.so.6")


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if a.size else 0.0


def _solve(impl, p, **kw):
    libc.srand(1)
    s = Qpalm(impl)
    st = dict(p.settings)
    st.update(kw)
    for k, v in st.items():
        setattr(s.settings, k, v)
    s.set_data(p.Q.copy(), p.A.copy(), p.q.copy(), p.bmin.copy(), p.bmax.copy())
    assert s._allocate_work()
    method = int(s.work.solver.contents.factorization_method)
    s._solve()
    r = s.result()
    stats = s.stats() if impl == "b200" else None
    s.cleanup()
    return r, stats, method


def _parity(g, r, tol=1e-8):
    assert g.status_val == r.status_val, (g.status, r.status)
    assert _rel(g.x, r.x) < tol and _rel(g.y, r.y) < tol, (_rel(g.x, r.x), _rel(g.y, r.y))
    assert abs(g.iter - r.iter) <= max(1, int(np.ceil(0.05 * r.iter))), (g.iter, r.iter)
    assert abs(g.iter_out - r.iter_out) <= max(1, int(np.ceil(0.05 * r.iter_out))), (g.iter_out, r.iter_out)


@pytest.mark.parametrize("make", [lambda: problems.grid_qp(12, seed=1), lambda: problems.grid_qp(24, seed=2),
                                  lambda: problems.random_qp(300, 600, 0.02, 0.01, seed=3),
                                  lambda: problems.grid_qp(18, seed=5, proximal=0, scaling=2)])
def test_forced_kkt_path_matches_the_reference(make):
    """settings.factorization_method = FACTORIZE_KKT (0): every Newton step through the L S L' factorization of the KKT matrix."""
    p = make()
    g, st, method = _solve("b200", p, factorization_method=0)
    assert method == 0 and st.kkt_factorizations > 0 and st.updown_calls == 0
    r, _, _ = _solve("reference" if HAS_REF else "oracle", p)
    _parity(g, r)
    # and the Schur path of this library on the same problem
    g2, st2, method2 = _solve("b200", p, factorization_method=1)
    assert method2 == 1 and st2.kkt_factorizations == 0
    _parity(g, g2)


def test_kkt_path_primal_infeasible_and_nonconvex():
    p = problems.prim_inf_qp()
    # tiny dense problems stay on the Schur path even when KKT is asked for (the KKT engine serves sparse data)
    g, st, _ = _solve("b200", p, factorization_method=0)
    assert g.status_val == -3
    q = problems.nonconvex_random_qp(400, 800, seed=2)
    g, st, method = _solve("b200", q, factorization_method=0)
    r, _, _ = _solve("oracle", q)
    assert g.status_val == r.status_val


@pytest.mark.timeout(900)
def test_schur_fill_in_problem_selects_kkt_automatically():
    """AUG2DCQP-class stand-in: coupling rows make Q + A'A dense; with DEFAULT settings the library must pick the KKT system by
    the reference's criterion (src/solver_interface.c:20-66), solve it to the gates, and be faster than its own dense Schur path."""
    import os
    import time
    os.environ["QPALM_B200_KKT_AUTO_MIN_N"] = "2048"   # the default threshold (6000) is where KKT starts to win; the reference run at that size takes minutes
    p = problems.kkt_standin_qp(2500, seed=0)
    t0 = time.perf_counter()
    g, st, method = _solve("b200", p)
    t_kkt = time.perf_counter() - t0
    assert method == 0 and st.kkt_factorizations > 0, "the KKT path was not selected"
    r, _, _ = _solve("reference" if HAS_REF else "oracle", p)
    _parity(g, r)
    t0 = time.perf_counter()
    g1, st1, method1 = _solve("b200", p, factorization_method=1)       # forced Schur: dense n x n factor
    t_schur = time.perf_counter() - t0
    assert st1.kkt_factorizations == 0
    _parity(g, g1)
    print(f"kkt_standin n=2500: KKT {t_kkt:.3f} s (nnz(L) {st.sparse_factor_nnz}, {st.kkt_factorizations} factorizations, "
          f"{st.kkt_refinement_steps} refinement steps) vs Schur (dense) {t_schur:.3f} s")


def test_forced_kkt_per_block_launches_equal_cluster_launches():
    """random_qp(300, 600) has fronts above the shared-memory size (263 rows at most): the per-block launches and the cluster
    launches of the signed factorization are bit-identical, so the whole trajectory must be too -- x, y, iteration counts
    and the number of iterative-refinement corrections."""
    import os
    p = problems.random_qp(300, 600, 0.02, 0.01, seed=3)
    out = {}
    for mode, flag in (("per_block", "1"), ("cluster", "0")):
        old = os.environ.get("QPALM_B200_MF_PER_BLOCK")
        os.environ["QPALM_B200_MF_PER_BLOCK"] = flag
        try:
            out[mode] = _solve("b200", p, factorization_method=0)
        finally:
            os.environ.pop("QPALM_B200_MF_PER_BLOCK", None) if old is None else os.environ.__setitem__("QPALM_B200_MF_PER_BLOCK", old)
    (a, sa, ma), (b, sb, mb) = out["per_block"], out["cluster"]
    assert ma == mb == 0 and sa.kkt_factorizations > 0
    assert np.array_equal(a.x, b.x) and np.array_equal(a.y, b.y)
    assert (a.iter, a.iter_out) == (b.iter, b.iter_out)
    assert (sa.kkt_factorizations, sa.kkt_refinement_steps) == (sb.kkt_factorizations, sb.kkt_refinement_steps)
    print(f"random_qp(300, 600) forced KKT: {a.iter} iterations, {sa.kkt_factorizations} factorizations, "
          f"{sa.kkt_refinement_steps} refinement corrections")
