"""The persistent batch engine's exact line search (batchp.cu: p_ls_build, p_ls_sort, p_ls_select), in both CTA shapes.

The sort orders only the breakpoints s > 0, so its real keys are bit patterns of positive doubles and +inf, nL <= 2m of
them, with exact ties that must keep their input order: the walk's running sums, and so tau, depend on that order.  The
solver-level case runs the benchmark's instance size in the build the benchmark selects and reads the line-search
counters (qpalm_b200_batch_linesearch_stats)."""
import numpy as np
import pytest

from qpalm_b200 import problems
from qpalm_b200 import batch as qb
from test_gpu_batch import _check_instances
from test_gpu_batch_cta import SHAPES, _sms, probe_sort

pytestmark = pytest.mark.gpu

INF = np.uint64(0x7FF0000000000000)
# nL-like sizes: around the register runs (8 per thread), the merge levels, one chunk of the walk (256), the benchmark's
# 2m = 1898 and the largest sort
LS_N = (1, 7, 8, 9, 16, 17, 100, 255, 256, 257, 513, 949, 1024, 1025, 1898, 2047, 2048)


def _breakpoints(rng, N, pool):
    """Positive doubles over 30 decades and +inf, drawn from `pool` distinct values so that exact ties are frequent."""
    vals = np.exp(rng.uniform(-35, 35, pool))
    vals[rng.random(pool) < 0.1] = np.inf
    return rng.choice(vals, N).view(np.uint64).copy()


@pytest.mark.parametrize("shape", SHAPES, ids=["shape3", "shape4"])
@pytest.mark.parametrize("pool", [4, 64, 100000], ids=["ties_heavy", "ties_some", "ties_rare"])
def test_sort_breakpoint_keys(shape, pool):
    """Each instance's sort against a stable argsort: keys ascending, equal keys by input position."""
    rng = np.random.default_rng(900 + pool % 97 + shape)
    for N in LS_N:
        keys = np.stack([_breakpoints(rng, N, pool) for _ in range(4)])
        keys[0, :] = INF   # every key tied
        vals = np.tile(np.arange(N, dtype=np.uint32), (4, 1))
        ks, vs = probe_sort(shape, keys, vals)
        for b in range(4):
            order = np.argsort(keys[b], kind="stable")
            assert np.array_equal(ks[b], keys[b][order]), (shape, pool, N, b)
            assert np.array_equal(vs[b], vals[b][order]), (shape, pool, N, b)


def test_benchmark_shape_against_oracle_and_counters():
    """The benchmark's instance size (n = 240, m = 949) with 3 SMs + 1 instances, so the 4-CTAs-per-SM build runs: sampled
    instances against the oracle, and the line-search counters within their bounds (the walk reads at most the sorted
    breakpoints, at most 2m of them per line search)."""
    nb = 3 * _sms() + 1
    b = problems.mpc_batch(nb, seed=7)
    h = qb.Batch(b.Q, b.A, b.settings, nb)
    assert h.ok
    try:
        xs, ys, infos = h.solve(b.q, b.bmin, b.bmax)
        assert h.last_shape() == 4
        st = h.stats(nb)
    finally:
        h.cleanup()
    m = b.A.nrow
    assert st["inner"] > 0
    assert 0 < st["ls_walked"] <= st["ls_breakpoints"] <= 2 * m * st["inner"], st
    worst = int(np.argmax([i["iter"] for i in infos]))
    _check_instances(b, sorted({0, nb // 2, nb - 1, worst}), xs, ys, infos)
