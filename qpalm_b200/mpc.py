"""Warm-started sequential MPC loop over one workspace (SURVEY.md 8(f4)).

The caller pattern either side of `qpalm_solve` in receding-horizon control (the reference's `examples/`, and
`qpalm_update_bounds` / `qpalm_update_q` / `qpalm_warm_start`, src/qpalm.c:322-399,793-871): set the problem up once,
then per time step change q and the bounds, warm-start from the previous primal/dual solution and solve again.  With the
B200 library the matrices, the scaling, the factor storage and every iterate stay resident in HBM between the steps; a
step moves only q, bmin, bmax (and the warm start) to the device and x, y back.
"""
from __future__ import annotations

import time

import numpy as np

from . import problems
from .interface import Qpalm


def mpc_sequence(steps: int, n: int = 240, m0: int = 709, seed: int = 0, drift: float = 0.01):
    """A base chain80w-sized instance and `steps` slowly drifting (q, bmin, bmax) triples."""
    b = problems.mpc_batch(1, n=n, m0=m0, seed=seed)
    rng = np.random.default_rng(seed + 12345)
    q, lo, hi = b.q[0].copy(), b.bmin[0].copy(), b.bmax[0].copy()
    seq = []
    for _ in range(steps):
        q = q + drift * rng.standard_normal(q.size)
        shift = drift * rng.standard_normal(lo.size)
        lo, hi = lo + shift, hi + shift
        seq.append((q.copy(), lo.copy(), hi.copy()))
    return b, seq


def batch_sequence(nb: int, steps: int, n: int = 240, m0: int = 709, seed: int = 0, drift: float = 0.01):
    """The batch form of mpc_sequence: a chain80w-sized BatchQP of nb instances and, per step, the (q, bmin, bmax) arrays
    (nb x n, nb x m, nb x m) of all instances.  Every instance drifts as mpc_sequence's does, from its own PRNG stream."""
    b = problems.mpc_batch(nb, n=n, m0=m0, seed=seed)
    rngs = [np.random.default_rng([seed + 12345, k]) for k in range(nb)]
    q, lo, hi = b.q.copy(), b.bmin.copy(), b.bmax.copy()
    seq = []
    for _ in range(steps):
        for k, rng in enumerate(rngs):
            q[k] = q[k] + drift * rng.standard_normal(q.shape[1])
            shift = drift * rng.standard_normal(lo.shape[1])
            lo[k], hi[k] = lo[k] + shift, hi[k] + shift
        seq.append((q.copy(), lo.copy(), hi.copy()))
    return b, seq


def run_sequence(impl: str, b, seq, warm: bool = True, **settings):
    """Returns (results, seconds per step) of the warm-started loop on one workspace."""
    s = Qpalm(impl)
    st = dict(b.settings)
    st.update(settings)
    for k, v in st.items():
        setattr(s.settings, k, v)
    s.set_data(b.Q.copy(), b.A.copy(), b.q[0].copy(), b.bmin[0].copy(), b.bmax[0].copy())
    if not s._allocate_work():
        raise RuntimeError("qpalm_setup returned NULL")
    s._solve()
    prev = s.result()
    out, times = [prev], []
    for (q, lo, hi) in seq:
        t0 = time.perf_counter()
        s._update_q(q)
        s._update_bounds(lo, hi)
        if warm:
            s._warm_start(prev.x, prev.y)
        s._solve()
        prev = s.result()
        times.append(time.perf_counter() - t0)
        out.append(prev)
    s.cleanup()
    return out, times
