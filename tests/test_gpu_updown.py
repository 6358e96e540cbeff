"""The cholmod_updown replacement on the dense Newton system (updown_gen.cu: generator-form passes of <= 32 columns) --
operator level against the oracle's restatement of CHOLMOD's recurrence (Modify/t_cholmod_updown_numkr.c:289-376)
and solver level: the rank-update branch of newton_set_direction (src/newton.c:96-108) and ldlupdate_sigma_changed
(src/solver_interface.c:443-503, caller src/iteration.c:135-144) must actually be TAKEN on the GPU, with the same
solutions and iteration counts as the reference."""
import ctypes

import numpy as np
import pytest

from conftest import HAS_REF
from qpalm_b200 import problems
from qpalm_b200.interface import Qpalm

pytestmark = pytest.mark.gpu
libc = ctypes.CDLL("libc.so.6")


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(1.0, np.max(np.abs(b))) if a.size else 0.0


@pytest.mark.parametrize("n,k", [(256, 1), (300, 33), (500, 9), (777, 64), (1000, 70), (1400, 40), (2304, 64), (3000, 150)])
def test_dataflow_rank_k_update_and_downdate(gpu_ops, oracle_ops, n, k):
    """L L' +- W W' for factors of >= 2 blocks (generator form: passes of <= 8 / 16 / 32 columns, k > 32 takes several)."""
    rng = np.random.default_rng(n + k)
    M = rng.standard_normal((n, n))
    H = M @ M.T + n * np.eye(n)
    L = np.linalg.cholesky(H)
    W = rng.standard_normal((n, k))
    Lu_g = gpu_ops.updown(L, W, 1)
    assert _rel(Lu_g @ Lu_g.T, H + W @ W.T) < 1e-12
    if n <= 1400:
        Lu_o = oracle_ops.updown(L, W, 1)
        assert _rel(Lu_g, Lu_o) < 1e-10
    assert np.all(np.diag(Lu_g) > 0) and np.allclose(np.triu(Lu_g, 1), 0.0)
    Ld_g = gpu_ops.updown(Lu_g, W, 0)
    assert _rel(Ld_g @ Ld_g.T, H) < 1e-12
    assert _rel(Ld_g, L) < 1e-9           # update then downdate is the identity


def test_mixed_update_downdate_pass_matches_cholesky():
    """Entering and leaving rows share a pass (S = diag(+1.., -1..)): solver-level check that a step with both kinds of
    change lands on the factor of the new matrix -- forced updates against forced refactorisations on a problem whose active
    set churns (the operator entry point only takes one sign per call)."""
    p = problems.random_qp(520, 1100, 1.0, 1.0, seed=21)
    g1, s1 = _solve("b200", p, max_rank_update=400, max_rank_update_fraction=1.0)
    g0, s0 = _solve("b200", p, max_rank_update=0)
    assert s1.updown_calls > 0 and s0.updown_calls == 0
    assert g1.status_val == g0.status_val == 1
    assert _rel(g1.x, g0.x) < 1e-8 and _rel(g1.y, g0.y) < 1e-8


def test_update_then_partial_downdate_matches_cholesky(gpu_ops):
    """A 24-column update followed by a downdate of 7 of those columns lands on the factor of H + W W' - W_7 W_7'."""
    n, k = 1152, 24
    rng = np.random.default_rng(5)
    M = rng.standard_normal((n, n)); H = M @ M.T + n * np.eye(n)
    L = np.linalg.cholesky(H); W = rng.standard_normal((n, k))
    Lg = gpu_ops.updown(gpu_ops.updown(L, W, 1), W[:, :7], 0)
    Href = H + W @ W.T - W[:, :7] @ W[:, :7].T
    assert _rel(Lg @ Lg.T, Href) < 1e-12


def test_downdate_that_loses_definiteness_is_reported(gpu_ops):
    """A downdate past positive definiteness must come back as an error code (the solver then refactorises), not hang."""
    n = 512
    L = np.linalg.cholesky(np.eye(n) * 4.0)
    W = np.zeros((n, 2))
    W[300, 0] = 3.0        # 4 - 9 < 0
    Lc, Wc = np.asfortranarray(L.copy()), np.asfortranarray(W.copy())
    from qpalm_b200 import abi
    rc = gpu_ops._updown(n, 2, Lc.ctypes.data_as(abi.c_float_p), Wc.ctypes.data_as(abi.c_float_p), 0)
    assert rc == 1000


def _solve(impl, p, **kw):
    libc.srand(1)
    s = Qpalm(impl)
    st = dict(p.settings)
    st.update(kw)
    for k, v in st.items():
        setattr(s.settings, k, v)
    s.set_data(p.Q.copy(), p.A.copy(), p.q.copy(), p.bmin.copy(), p.bmax.copy())
    assert s._allocate_work()
    s._solve()
    r = s.result()
    stats = s.stats() if impl == "b200" else None
    s.cleanup()
    return r, stats


def _parity(g, r, tol=1e-8, iter_tol=0.05):
    assert g.status_val == r.status_val == 1, (g.status, r.status)
    assert _rel(g.x, r.x) < tol and _rel(g.y, r.y) < tol, (_rel(g.x, r.x), _rel(g.y, r.y))
    assert abs(g.iter - r.iter) <= max(1, int(np.ceil(iter_tol * r.iter))), (g.iter, r.iter)
    assert abs(g.iter_out - r.iter_out) <= max(1, int(np.ceil(iter_tol * r.iter_out))), (g.iter_out, r.iter_out)


@pytest.mark.parametrize("n,m,dA,dM,seed", [(600, 1200, 1.0, 1.0, 3), (1000, 2000, 0.3, 1.0, 4), (400, 900, 1.0, 1.0, 6)])
def test_rank_update_branch_is_taken_with_default_settings(n, m, dA, dM, seed):
    """newton.c:98-108 with the DEFAULT settings (max_rank_update 160, fraction 0.1): the GPU must take rank updates where the
    reference does (updown_calls > 0) and land on the same solution / iteration counts."""
    p = problems.random_qp(n, m, dA, dM, seed=seed)
    g, st = _solve("b200", p)
    r, _ = _solve("reference" if HAS_REF else "oracle", p)
    _parity(g, r)
    assert st.updown_calls > 0 and st.updown_rank_sum > 0, (st.updown_calls, st.refactorizations)
    assert st.refactorizations < g.iter        # not one refactorisation per iteration any more


def test_sigma_changed_update_is_taken():
    """a10 ldlupdate_sigma_changed: with gamma at gamma_max from the start (default settings) a small number of sigma changes at
    an outer iteration is absorbed by a rank update; assert the branch ran and parity holds."""
    hit = 0
    for seed in (3, 4, 6, 11):
        p = problems.random_qp(500, 1000, 1.0, 1.0, seed=seed)
        g, st = _solve("b200", p)
        r, _ = _solve("reference" if HAS_REF else "oracle", p)
        _parity(g, r)
        hit += int(st.sigma_update_calls > 0)
        if st.sigma_update_calls > 0:
            assert st.sigma_update_rank_sum <= 40 * st.sigma_update_calls       # iteration.c:136: at most 0.25 * max_rank_update rows
    assert hit > 0, "no instance took the sigma-changed rank update"


def test_forced_updates_match_forced_refactorisations():
    """Same matrix either way: with every eligible step forced through the update sweep (max_rank_update_fraction = 1, rank limit
    raised) the solution equals the refactorise-always run."""
    p = problems.random_qp(700, 1400, 1.0, 1.0, seed=9)
    g1, s1 = _solve("b200", p, max_rank_update=400, max_rank_update_fraction=1.0)
    g0, s0 = _solve("b200", p, max_rank_update=0)
    assert s1.updown_calls > 0 and s0.updown_calls == 0
    assert g1.status_val == g0.status_val == 1
    assert _rel(g1.x, g0.x) < 1e-8 and _rel(g1.y, g0.y) < 1e-8
