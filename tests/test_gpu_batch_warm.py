"""Per-instance warm starts of the batch entry point (qpalm_b200_batch_warm_start): instance k of a warm-started batch must
equal what qpalm_setup + qpalm_warm_start(x_ws[k], y_ws[k]) + qpalm_solve return for that instance alone, with the gates of
test_gpu_batch._check_instances.  Every case runs on the lock-step engine and on the persistent one in both CTA shapes
(3 per SM for small batches, 4 per SM for 3 SMs < nb <= 4 SMs instances, asserted with last_shape); a zero warm start and
the instances outside a warm start must be bit-identical to a cold solve."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from qpalm_b200 import batch as qb
from qpalm_b200 import mpc, problems
from qpalm_b200.abi import fptr
from qpalm_b200.interface import solve_qp

pytestmark = pytest.mark.gpu

SETTINGS = {
    "chain80w": (dict(n=48, m0=80), {}),
    "scaling0": (dict(n=48, m0=80), dict(scaling=0)),
    "scaling10_proximal": (dict(n=40, m0=60), dict(scaling=10, proximal=1, eps_abs_in=1.0, eps_rel_in=1.0, eps_prim_inf=1e-5,
                                                   eps_dual_inf=1e-5)),
}
MODES = ["xy", "x", "y"]


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(params=[("lockstep", 0), ("persistent", 3), ("persistent", 4)], ids=["lockstep", "persistent3", "persistent4"])
def engine(request, monkeypatch):
    """(engine, shape); the persistent shape follows from nb, as for a user: see _nb."""
    monkeypatch.setenv("QPALM_B200_BATCH_ENGINE", request.param[0])
    return request.param


def _nb(engine, small=6):
    return 3 * _sms() + 1 if engine[1] == 4 else small


def _sample(nb):
    return sorted({0, 1, nb // 2, nb - 1})


def _rel(a, b):
    return np.max(np.abs(a - b)) / max(1.0, np.max(np.abs(b))) if a.size else 0.0


def _perturbed(b, seed, scale=0.05):
    r = np.random.default_rng(seed)
    shift = scale * r.standard_normal(b.bmin.shape)
    return dataclasses.replace(b, q=b.q + scale * r.standard_normal(b.q.shape), bmin=b.bmin + shift, bmax=b.bmax + shift)


def _ws(mode, xs, ys):
    return (xs if "x" in mode else None), (ys if "y" in mode else None)


def _solve(b, engine, x_ws=None, y_ws=None):
    h = qb.Batch(b.Q, b.A, b.settings, b.q.shape[0])
    assert h.ok
    try:
        out = h.solve(b.q, b.bmin, b.bmax, x_ws=x_ws, y_ws=y_ws)
        assert h.last_shape() == engine[1]
    finally:
        h.cleanup()
    return out


def _check_warm(b, idx, xs, ys, infos, x_ws, y_ws, tol=1e-7):
    """Instances idx against the oracle's setup + warm start + solve (test_gpu_batch._check_instances gates)."""
    iters = []
    for k in idx:
        q = b.instance(k)
        o = solve_qp("oracle", q.Q.copy(), q.A.copy(), q.q, q.bmin, q.bmax,
                     warm_x=None if x_ws is None else x_ws[k].copy(), warm_y=None if y_ws is None else y_ws[k].copy(), **q.settings)
        g = infos[k]
        assert g["status_val"] == o.status_val, (k, g, o.status)
        assert abs(g["iter"] - o.iter) <= max(1, int(np.ceil(0.05 * o.iter))), (k, g["iter"], o.iter)
        assert abs(g["iter_out"] - o.iter_out) <= 1, (k, g["iter_out"], o.iter_out)
        if o.status_val == 1:
            assert _rel(xs[k], o.x) < tol, (k, _rel(xs[k], o.x))
            assert _rel(ys[k], o.y) < tol, (k, _rel(ys[k], o.y))
            assert abs(g["objective"] - o.objective) <= 1e-7 * max(1.0, abs(o.objective))
        iters.append((g["iter"], o.iter))
    return iters


def _same(a, b, rows):
    """Bit-identical x, y and info on the given instances."""
    for k in rows:
        assert np.array_equal(a[0][k], b[0][k]) and np.array_equal(a[1][k], b[1][k]), k
        assert a[2][k] == b[2][k], (k, a[2][k], b[2][k])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", list(SETTINGS))
def test_warm_start_matches_single_qp_contract(engine, case, mode):
    shape_kw, st = SETTINGS[case]
    nb = _nb(engine)
    b = problems.mpc_batch(nb, seed=3, **shape_kw, **st)
    xs0, ys0, _ = _solve(_perturbed(b, 17), engine)
    x_ws, y_ws = _ws(mode, xs0, ys0)
    xs, ys, infos = _solve(b, engine, x_ws, y_ws)
    _check_warm(b, _sample(nb), xs, ys, infos, x_ws, y_ws)


def test_resolve_from_own_solution(engine):
    nb = _nb(engine)
    b = problems.mpc_batch(nb, n=48, m0=80, seed=5)
    xs0, ys0, cold = _solve(b, engine)
    xs, ys, infos = _solve(b, engine, xs0, ys0)
    for g, o in _check_warm(b, _sample(nb), xs, ys, infos, xs0, ys0):
        assert g <= 12, (g, o)   # tests/src/test_basic_qp.c:202 pins iter < 12 after a warm start from the solution
    assert max(i["iter"] for i in infos) < min(i["iter"] for i in cold)


def test_zero_warm_start_is_a_cold_start(engine):
    nb = _nb(engine)
    b = problems.mpc_batch(nb, n=48, m0=80, seed=7)
    cold = _solve(b, engine)
    warm = _solve(b, engine, np.zeros((nb, b.Q.ncol)), np.zeros((nb, b.A.nrow)))
    _same(cold, warm, range(nb))


def test_mixed_zero_and_warm_rows(engine):
    nb = _nb(engine)
    b = problems.mpc_batch(nb, n=48, m0=80, seed=8)
    cold = _solve(b, engine)
    xs0, ys0, _ = _solve(_perturbed(b, 18), engine)
    x_ws, y_ws = xs0.copy(), ys0.copy()
    x_ws[0::2] = 0.0
    y_ws[0::2] = 0.0
    out = _solve(b, engine, x_ws, y_ws)
    _same(cold, out, range(0, nb, 2))
    _check_warm(b, sorted({k | 1 for k in _sample(nb)} & set(range(nb))), *out, x_ws, y_ws)   # odd rows: warm


def test_pending_state(engine):
    nb = _nb(engine)
    b = problems.mpc_batch(nb, n=48, m0=80, seed=9)
    xs0, ys0, _ = _solve(_perturbed(b, 19), engine)
    h = qb.Batch(b.Q, b.A, b.settings, nb)
    assert h.ok
    try:
        cold = h.solve(b.q, b.bmin, b.bmax)
        half = nb // 2
        part = h.solve(b.q, b.bmin, b.bmax, x_ws=xs0[:half], y_ws=ys0[:half])
        assert h.last_shape() == engine[1]
        _same(cold, part, range(half, nb))
        assert part[2][0] != cold[2][0] or not np.array_equal(part[0][0], cold[0][0])
        _same(cold, h.solve(b.q, b.bmin, b.bmax), range(nb))          # consumed by the solve
        h.warm_start(xs0, ys0)
        h.warm_start()                                                  # (NULL, NULL) clears it
        _same(cold, h.solve(b.q, b.bmin, b.bmax), range(nb))
        full = h.solve(b.q, b.bmin, b.bmax, x_ws=xs0, y_ws=ys0)
        h.warm_start(xs0, ys0)
        for bad in (0, nb + 1, -1):                                     # invalid nb: 1, the pending warm start stays
            assert h.lib.qpalm_b200_batch_warm_start(h.h, bad, fptr(xs0), fptr(ys0)) == 1
        _same(full, h.solve(b.q, b.bmin, b.bmax), range(nb))
        with pytest.raises(ValueError):
            h.warm_start(np.zeros((nb, b.Q.ncol + 1)))
        with pytest.raises(ValueError):
            h.warm_start(y=np.zeros((nb + 1, b.A.nrow)))
    finally:
        h.cleanup()


def test_receding_horizon(engine):
    nb = _nb(engine, small=5)
    b, seq = mpc.batch_sequence(nb, 4, n=48, m0=80, seed=2, drift=0.01)
    prev = _solve(b, engine)
    for step, (q, lo, hi) in enumerate(seq):
        bs = dataclasses.replace(b, q=q, bmin=lo, bmax=hi)
        out = _solve(bs, engine, prev[0], prev[1])
        _check_warm(bs, _sample(nb), *out, prev[0], prev[1])
        prev = out


def test_chain80w_size_shape4(monkeypatch):
    engine = ("persistent", 4)
    monkeypatch.setenv("QPALM_B200_BATCH_ENGINE", engine[0])
    nb = _nb(engine)
    b = problems.mpc_batch(nb, seed=1)
    xs0, ys0, _ = _solve(_perturbed(b, 21, scale=0.01), engine)
    out = _solve(b, engine, xs0, ys0)
    _check_warm(b, [0, nb // 2, nb - 1], *out, xs0, ys0)
