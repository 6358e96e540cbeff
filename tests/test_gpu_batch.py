"""Batch entry point (BASELINE config 4): every instance of a batch must equal what qpalm_setup + qpalm_solve return for
that instance alone (SURVEY.md 8(b) "Batch entry point") -- checked against the oracle per instance."""
import numpy as np
import pytest

from qpalm_b200 import batch as qb
from qpalm_b200 import problems
from qpalm_b200.interface import solve_qp

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(1.0, np.max(np.abs(b))) if a.size else 0.0


@pytest.fixture(params=["persistent", "lockstep"], autouse=True)
def engine(request, monkeypatch):
    """Both batch engines are exercised: the persistent one-CTA-per-instance kernel (batchp.cu, default whenever the
    shapes fit) and the lock-step engine (batch.cu, any size)."""
    monkeypatch.setenv("QPALM_B200_BATCH_ENGINE", request.param)
    return request.param


def _check_batch(b, idx, tol=1e-7):
    xs, ys, infos = qb.solve_batch(b)
    _check_instances(b, idx, xs, ys, infos, tol)
    return xs, ys, infos


def _check_instances(b, idx, xs, ys, infos, tol=1e-7):
    """Instances idx of a solved batch against the oracle: status, iteration counts, x, y and objective."""
    for k in idx:
        q = b.instance(k)
        o = solve_qp("oracle", q.Q.copy(), q.A.copy(), q.q, q.bmin, q.bmax, **q.settings)
        g = infos[k]
        assert g["status_val"] == o.status_val, (k, g, o.status)
        assert abs(g["iter"] - o.iter) <= max(1, int(np.ceil(0.05 * o.iter))), (k, g["iter"], o.iter)
        assert abs(g["iter_out"] - o.iter_out) <= 1, (k, g["iter_out"], o.iter_out)
        if o.status_val == 1:
            assert _rel(xs[k], o.x) < tol, (k, _rel(xs[k], o.x))
            assert _rel(ys[k], o.y) < tol, (k, _rel(ys[k], o.y))
            assert abs(g["objective"] - o.objective) <= 1e-7 * max(1.0, abs(o.objective))


def test_batch_small_chain80w_settings():
    """scaling=2, proximal=FALSE, eps_*_in = 1 (simulations/chain80w.m:39-51)."""
    _check_batch(problems.mpc_batch(12, n=48, m0=80, seed=3), range(12))


def test_batch_default_settings_proximal_and_boost():
    """Reference defaults (scaling 10, proximal, gamma_init = gamma_max = 1e7): exercises update/boost_gamma."""
    b = problems.mpc_batch(6, n=40, m0=60, seed=5, scaling=10, proximal=1, eps_abs_in=1.0, eps_rel_in=1.0,
                           eps_prim_inf=1e-5, eps_dual_inf=1e-5)
    _check_batch(b, range(6))
    b2 = problems.mpc_batch(4, n=40, m0=60, seed=6, scaling=0, proximal=1, gamma_init=1e1, gamma_max=1e7)
    _check_batch(b2, range(4))


def test_batch_chain80w_size():
    """n=240, m=949 (BASELINE config 4 instance size)."""
    _check_batch(problems.mpc_batch(6, seed=1), [0, 3, 5])


def test_batch_with_infeasible_instance():
    b = problems.mpc_batch(5, n=30, m0=40, seed=9)
    b.bmin[2, :] = 5.0      # row bounds [5, 6] on both A0 x and x itself cannot all hold -> primal infeasible
    b.bmax[2, :] = 6.0
    b.bmin[2, 0], b.bmax[2, 0] = -9.0, -8.0
    xs, ys, infos = _check_batch(b, range(5))
    assert infos[2]["status_val"] in (-3, -2)


def test_batch_is_deterministic():
    b = problems.mpc_batch(8, n=48, m0=80, seed=11)
    x1, y1, i1 = qb.solve_batch(b)
    x2, y2, i2 = qb.solve_batch(b)
    assert np.array_equal(x1, x2) and np.array_equal(y1, y2)
    assert [i["iter"] for i in i1] == [i["iter"] for i in i2]


@pytest.mark.parametrize("cap", ["0", "8", "1000000"], ids=["refactorize_always", "one_sweep", "sweeps_always"])
def test_batch_update_and_refactorization_paths_agree(cap, monkeypatch, engine):
    """Same matrix either way: the persistent engine's in-CTA update sweeps (chain warp + row owners) against its incremental
    SYRK + refactorization, selected through the rank cap (default 40).  Every instance must land on the oracle's solution
    and iteration count whichever path its Newton systems took, and the sweep path must actually have run."""
    if engine != "persistent":
        pytest.skip("the lock-step engine always refactorizes")
    monkeypatch.setenv("QPALM_B200_BATCH_UPDOWN_MAX_RANK", cap)
    b = problems.mpc_batch(5, n=61, m0=90, seed=21)      # 61 columns: three full 16-column blocks + a ragged one, rows beyond the 32-row window
    h = qb.Batch(b.Q, b.A, b.settings, 5)
    xs, ys, infos = h.solve(b.q, b.bmin, b.bmax)
    st = h.stats(5)
    h.cleanup()
    assert (st["updown_sweeps"] > 0) == (cap != "0"), st
    assert st["updown_failed"] == 0
    for k in range(5):
        q = b.instance(k)
        o = solve_qp("oracle", q.Q.copy(), q.A.copy(), q.q, q.bmin, q.bmax, **q.settings)
        assert infos[k]["status_val"] == o.status_val == 1
        assert abs(infos[k]["iter"] - o.iter) <= max(1, int(np.ceil(0.05 * o.iter))), (k, infos[k]["iter"], o.iter)
        assert _rel(xs[k], o.x) < 1e-7 and _rel(ys[k], o.y) < 1e-7
