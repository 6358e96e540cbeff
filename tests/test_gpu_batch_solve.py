"""The persistent batch engine's triangular solves (batchp.cu, cta_chol_solve) in both CTA shapes, over many rounds per instance.

The solves run as a dataflow on the update sweep's per-column mbarriers: a chain warp on the diagonal and one owner per entry
of v, each mbarrier completing one phase per 16-column block.  The phase carries across solves, sweeps and the instances a
persistent CTA takes, so the probe (qpalm_b200_batchp_probe_solves) runs, per instance, `rounds` rounds of {update sweeps,
solve} and then `rounds` rounds of {solve}, and every round's d is checked against its float64 bound.  n covers one entry,
the 16-column blocks of the solve, the panels of the factorisation and the engine's largest n."""
import ctypes as C

import numpy as np
import pytest

from qpalm_b200 import abi
from test_gpu_batch_cta import _grid, _lib, base, check_solve, gram, updated_bound

pytestmark = pytest.mark.gpu

SHAPES = (3, 4)
SOLVE_N = (1, 2, 15, 16, 17, 23, 24, 25, 31, 32, 33, 47, 48, 49, 96, 97, 223, 239, 240)
ROUNDS = 3


@pytest.fixture(params=SHAPES, ids=["shape3", "shape4"])
def shape(request):
    return request.param


def probe_solves(shape, A, insts, rounds):
    """insts: dicts with H0 (n x n SPD), rhs and upd = (rows, weights).  Returns d_fused (the solve right after the
    factorisation) and the rounds' d (nb x 2 rounds x n)."""
    lib = _lib()
    if not getattr(lib, "_probe_solves_typed", False):
        fp, ip, ci = abi.c_float_p, abi.c_int_p, abi.c_int
        lib.qpalm_b200_batchp_probe_solves.argtypes = [ci, ci, ci, ci, fp, fp, ci, C.c_double, ip, ip, fp, C.c_double, fp,
                                                       fp, fp, fp, fp, ip, ci, fp]
        lib.qpalm_b200_batchp_probe_solves.restype = C.c_int
        lib._probe_solves_typed = True
    A = np.ascontiguousarray(A, dtype=np.float64)
    m, n = A.shape
    nb = len(insts)
    cnt = np.zeros((nb, 4), np.int64)
    lists = np.zeros((nb, 3, m), np.int64)
    wts = np.zeros((nb, 3, m))
    for b, it in enumerate(insts):
        rows, w = it["upd"]
        cnt[b, 2] = len(rows)   # the probe's own update (before the rounds) is all leaving: kpos = 0 -- see _instance
        lists[b, 2, :len(rows)] = rows
        wts[b, 2, :len(rows)] = w
    H0 = np.ascontiguousarray(np.stack([it["H0"].T for it in insts]), dtype=np.float64)
    rhs = np.ascontiguousarray(np.stack([it["rhs"] for it in insts]), dtype=np.float64)
    H, L = np.zeros((nb, n, n)), np.zeros((nb, n, n))
    dfu, daf = np.zeros((nb, n)), np.zeros((nb, n))
    info = np.zeros(nb, np.int64)
    dr = np.zeros((nb, 2 * rounds, n))
    rc = lib.qpalm_b200_batchp_probe_solves(shape, nb, n, m, abi.fptr(A), abi.fptr(H0), 0, 1.0, abi.iptr(cnt), abi.iptr(lists),
                                            abi.fptr(wts), 0.0, abi.fptr(rhs), abi.fptr(H), abi.fptr(L), abi.fptr(dfu),
                                            abi.fptr(daf), abi.iptr(info), rounds, abi.fptr(dr))
    assert rc == 0, rc
    assert not np.any(info), info
    return dfu, dr


def _instance(rng, A, n, k):
    """H0 = B + W'W: the probe first takes the k rows out (a downdate to B), then every even round puts them back and every
    odd round takes them out again."""
    m = A.shape[0]
    rows, w = rng.choice(m, k, replace=False), rng.uniform(0.5, 1.5, k)
    B = base(rng, n)
    G = gram(A, rows, w)
    return dict(H0=B + G, B=B, G=G, upd=(rows, w), rhs=rng.standard_normal(n))


def _check_rounds(it, dfu, dr, rounds, what):
    n = len(it["rhs"])
    H0, B, G = it["H0"], it["B"], it["G"]
    check_solve(dfu, H0, np.linalg.cholesky(H0), it["rhs"], what + ("fused",))
    k = len(it["upd"][0])
    S = np.max(np.diag(H0))
    for r in range(2 * rounds):
        s = min(r, rounds - 1)   # the last update round before this solve
        M = B + G if s % 2 == 0 else B
        dM = updated_bound(n, k * (s + 2), S)   # ranks swept so far: the probe's downdate and one pass per update round
        check_solve(dr[r], M, np.linalg.cholesky(M), (r + 1) * it["rhs"], what + ("round", r), dM=dM)


@pytest.mark.parametrize("n", SOLVE_N)
def test_solve_rounds(shape, n):
    """Per instance: factor, solve; downdate, solve; then rounds of {update / downdate sweeps, solve} and rounds of {solve}.
    Several instances with different update ranks (0, 1, 8, 13) share the launch, so CTAs take instances whose blocks and
    sweeps leave the mbarriers at different phases."""
    rng = np.random.default_rng(700 + n)
    m = 40
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    insts = [_instance(rng, A, n, k) for k in (0, 1, 8, 13)]
    dfu, dr = probe_solves(shape, A, insts, ROUNDS)
    for b, it in enumerate(insts):
        _check_rounds(it, dfu[b], dr[b], ROUNDS, (n, b))


def test_identical_instances_give_identical_solves(shape):
    """2 grid + 3 copies of one instance at the benchmark's n: every round of every copy must give the same bits, whichever
    CTA and mbarrier phase it met."""
    n, m = 240, 60
    nb = 2 * _grid(shape) + 3
    rng = np.random.default_rng(800 + shape)
    A = rng.standard_normal((m, n)) / np.sqrt(n)
    it = _instance(rng, A, n, 11)
    dfu, dr = probe_solves(shape, A, [it] * nb, ROUNDS)
    assert all(np.array_equal(dfu[b], dfu[0]) for b in range(1, nb))
    assert all(np.array_equal(dr[b], dr[0]) for b in range(1, nb))
    _check_rounds(it, dfu[0], dr[0], ROUNDS, ("identical",))
