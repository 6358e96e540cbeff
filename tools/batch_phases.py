#!/usr/bin/env python
"""Per-phase SM-clock breakdown of the persistent batch engine (QPALM_B200_BATCH_PROF=1)."""
import ctypes as C
import os
import sys
os.environ["QPALM_B200_BATCH_PROF"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from qpalm_b200 import batch as qb, problems

nb = int(sys.argv[1]) if len(sys.argv) > 1 else 512
b = problems.mpc_batch(nb, seed=0)
h = qb.Batch(b.Q, b.A, b.settings, nb)
h.upload(b.q, b.bmin, b.bmax)
for _ in range(2):
    ms = h.solve_resident(nb)
out = np.zeros((nb, 32), dtype=np.int64)
h.lib.qpalm_b200_batch_phase_profile.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
assert h.lib.qpalm_b200_batch_phase_profile(h.h, nb, out.ctypes.data) == 0
x, y, infos = h.download(nb)
iters = np.array([i["iter"] for i in infos])
names = ["init", "res_m", "gemv_Atyh", "res_n+control", "outer/sigma/boost", "lists", "H syrk", "potrf", "solve", "gemv Qd+Ad",
         "ls_build", "sort", "select+update", "gemv Qd", "rank-k update sweeps", "H syrk: A' gather + stage wait", "potrf: panel load", "potrf: diag16", "potrf: solve16", "potrf: update16",
         "potrf: store", "potrf: trailing", "sweep: gather W", "sweep chain warp: block prologue", "sweep: whole block loop (row owner's clock)", "sweep chain warp: column loop",
         "sweep chain warp: block epilogue", "sweep chain warp: wait for the row owners",
         "solve fwd chain warp: column loop", "solve fwd chain warp: block ends + window waits",
         "solve bwd chain warp: column loop", "solve bwd chain warp: block ends + window waits"]
tot = out[:, :15].sum(axis=1)   # slots 15 .. 31 split phases 6 .. 8 and 14
print(f"nb={nb} solve {ms:.2f} ms; mean iters {iters.mean():.1f} max {iters.max()}; mean clocks/instance {tot.mean():.3e} ({tot.mean()/1.965e3:.0f} us)")
st = h.stats(nb)
print(f"per instance: refactorizations {st['refactorizations']/nb:.1f}, update sweeps {st['updown_sweeps']/nb:.1f} (ranks {st['updown_rank_sum']/nb:.1f}, failed {st['updown_failed']/nb:.2f}), inner {st['inner']/nb:.1f}")
nr = max(st["refactorizations"], 1)
print(f"H syrk: {st['syrk_entries']/nr:.1f} list entries per refactorization, scratch rebuilds {st['scratch_rebuilds']/nb:.1f} "
      f"per instance ({100*st['scratch_rebuilds']/nr:.0f}% of the refactorizations)")
nls = max(st["inner"], 1)
print(f"line search: {st['ls_breakpoints']/nls:.1f} breakpoints sorted (s > 0 of 2m = {2*b.A.nrow}), {st['ls_walked']/nls:.1f} walked, "
      f"per line search ({100*st['ls_walked']/max(st['ls_breakpoints'], 1):.1f}% of the sorted ones)")
for k in list(range(32)):
    print(f"{names[k]:22s} {out[:,k].mean()/1.965e3:10.1f} us/instance  {100*out[:,k].sum()/tot.sum():6.2f}%   per-iter {out[:,k].sum()/iters.sum()/1.965e3:7.2f} us")
