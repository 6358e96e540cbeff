"""Host side of the batch warm start (no GPU): the shape checks of Batch.warm_start and the receding-horizon sequence
generator mpc.batch_sequence."""
import numpy as np
import pytest

from qpalm_b200 import batch as qb
from qpalm_b200 import mpc


class _Lib:
    def __init__(self):
        self.calls = []

    def qpalm_b200_batch_warm_start(self, h, nb, x, y):
        self.calls.append((nb, x is not None, y is not None))
        return 0


def _batch(n=4, m=6, nb_max=3):
    b = object.__new__(qb.Batch)   # no device: only the host-side checks run
    b.lib, b.h, b.n, b.m, b.nb_max = _Lib(), None, n, m, nb_max
    return b


def test_warm_start_shape_checks():
    b = _batch()
    with pytest.raises(ValueError):
        b.warm_start(np.zeros((2, 5)))                      # wrong column count
    with pytest.raises(ValueError):
        b.warm_start(y=np.zeros((2, 7)))
    with pytest.raises(ValueError):
        b.warm_start(np.zeros((4, 4)))                      # more rows than nb_max
    with pytest.raises(ValueError):
        b.warm_start(np.zeros((2, 4)), np.zeros((3, 6)))    # x and y disagree
    with pytest.raises(ValueError):
        b.warm_start(np.zeros(4))
    assert b.lib.calls == []
    b.warm_start(np.zeros((2, 4)))
    b.warm_start(y=np.zeros((3, 6)))
    b.warm_start()
    assert b.lib.calls == [(2, True, False), (3, False, True), (0, False, False)]


def test_batch_sequence_drifts_each_instance_on_its_own_stream():
    b, seq = mpc.batch_sequence(4, 3, n=12, m0=10, seed=1, drift=0.01)
    assert len(seq) == 3
    prev = (b.q, b.bmin, b.bmax)
    for q, lo, hi in seq:
        assert q.shape == (4, 12) and lo.shape == hi.shape == (4, 22)
        assert np.allclose(hi - lo, b.bmax - b.bmin)        # bounds shift together, as in mpc_sequence
        assert 0 < np.max(np.abs(q - prev[0])) < 0.1
        prev = (q, lo, hi)
    b2, seq2 = mpc.batch_sequence(2, 3, n=12, m0=10, seed=1, drift=0.01)
    for (q, lo, hi), (q2, lo2, hi2) in zip(seq, seq2):   # instance k does not depend on nb
        assert np.array_equal(q[:2], q2) and np.array_equal(lo[:2], lo2) and np.array_equal(hi[:2], hi2)
