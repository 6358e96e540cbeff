#!/usr/bin/env python
"""Compare two `bench.py --dump-outputs DIR` dumps of the same seeded workload (not a test; run by hand).

    python tests/compare_bench_outputs.py PARENT_DIR NEW_DIR [--rtol 1e-8]

Checks that every QP (and the dense block, prefix dense_) ends with the same status_val, that x and y agree per QP within
rtol relative to max(1, max|.|) of the parent's row, and lists the per-QP differences in iteration count with the mean of
each side.  A change that only reorders floating-point sums must pass it; exit status 1 otherwise."""
import argparse
import os
import sys

import numpy as np


def load(d, name):
    p = os.path.join(d, name + ".npy")
    return np.load(p) if os.path.exists(p) else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("parent")
    ap.add_argument("new")
    ap.add_argument("--rtol", type=float, default=1e-8)
    a = ap.parse_args()
    ok = True
    for pre in ("", "dense_"):
        st0, st1 = load(a.parent, pre + "status_val"), load(a.new, pre + "status_val")
        if st0 is None:
            continue
        label = pre.rstrip("_") or "batch"
        same = np.array_equal(st0, st1)
        ok &= same
        print(f"[{label}] {len(st0)} QPs, status_val identical: {same}")
        for v in ("x", "y"):
            X0, X1 = np.atleast_2d(load(a.parent, pre + v)), np.atleast_2d(load(a.new, pre + v))
            rel = np.max(np.abs(X1 - X0), axis=1) / np.maximum(1.0, np.max(np.abs(X0), axis=1))
            print(f"[{label}] {v}: max relative difference {rel.max():.3e} (QP {int(rel.argmax())}), within {a.rtol:g}: {bool(rel.max() <= a.rtol)}")
            ok &= bool(rel.max() <= a.rtol)
        it0, it1 = load(a.parent, pre + "iter"), load(a.new, pre + "iter")
        d = (it1 - it0).astype(np.int64)
        print(f"[{label}] mean iterations {it0.mean():.4f} -> {it1.mean():.4f} ({100 * (it1.mean() / it0.mean() - 1):+.3f} %)")
        nz = np.nonzero(d)[0]
        print(f"[{label}] iteration differences: {len(nz)} QPs differ" + "".join(f"\n    QP {i}: {int(it0[i])} -> {int(it1[i])}" for i in nz))
    print("PASS" if ok else "FAIL")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
