"""The batch engine's in-CTA Cholesky on matrices that are not positive definite, in both CTA shapes.

A non-positive pivot anywhere in a panel -- in its first, second or third 8-column range, in the first or a later panel --
must set the factorization's info bit, end the factorization without a hang (the chain warp keeps publishing its columns,
so the row owners never wait on a column that does not come), and leave the healthy instances of the same launch exact."""
import numpy as np
import pytest

from test_gpu_batch_cta import check_factor, probe_newton, shape, spd  # noqa: F401  (shape: the fixture)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n", [33, 64, 97, 240])
def test_non_positive_pivot_sets_info(shape, n):
    rng = np.random.default_rng(700 + n)
    A = rng.standard_normal((4, n))
    cols = [k for k in (0, 5, 12, 20, 31, 40, 57, 90, 200, n - 1) if k < n]
    insts, bad = [], []
    for k in cols:
        for broken in (True, False):
            H = spd(rng, n, 1e3)
            if broken:   # the leading (k + 1) x (k + 1) block is indefinite: pivot k is the first non-positive one
                H[k, k] = -1.0
            insts.append(dict(H0=H, rhs=rng.standard_normal(n)))
            bad.append(broken)
    H, L, dfu, daf, info = probe_newton(shape, A, insts)
    for b, (it, broken) in enumerate(zip(insts, bad)):
        what = (n, cols[b // 2], broken)
        if broken:
            assert info[b] == 2, what
        else:
            assert info[b] == 0, what
            check_factor(L[b], it["H0"], what)
