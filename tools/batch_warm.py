"""Warm starts of the batch entry point over a receding-horizon sequence: cold against warm x+y, x only and y only.

    python tools/batch_warm.py --out DIR [--nb 512] [--steps 5] [--drifts 0.001,0.01]

512 chain80w-sized instances (n = 240, m = 949, one GPU's share of the BASELINE sweep) drift step by step as
mpc.batch_sequence makes them.  Every mode warm-starts from its own previous step (all start from one cold solve of the
base batch), and the modes alternate within a step, in a rotating order, so that they share the machine's state.  Per mode
and drift: device ms per step (solve_resident's event time: the solve kernels alone, no copies), mean and max iterations (a
one-wave launch ends with its slowest instance), the solved count and the persistent CTA shape.  The card's name and power
limit are read in the same run.  Writes DIR/batch_warm.json and prints it."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from qpalm_b200 import batch as qb  # noqa: E402
from qpalm_b200 import mpc  # noqa: E402

MODES = ("cold", "xy", "x", "y")


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                       check=True)
    name, power = (s.strip() for s in r.stdout.splitlines()[0].split(","))
    return name, power


def run_drift(nb, steps, drift, seed):
    b, seq = mpc.batch_sequence(nb, steps, seed=seed, drift=drift)
    h = qb.Batch(b.Q, b.A, b.settings, nb)
    if not h.ok:
        raise RuntimeError("batch setup failed")
    try:
        for _ in range(2):   # warm-up: module load, first-touch of the per-instance buffers; the second one is step 0
            h.upload(b.q, b.bmin, b.bmax)
            h.solve_resident(nb)
        x0, y0, _ = h.download(nb)
        h.warm_start(x0[:1], y0[:1])   # and the warm path once (one instance warm)
        h.solve_resident(nb)
        prev = {mode: (x0, y0) for mode in MODES}
        rec = {mode: dict(ms=[], iter_mean=[], iter_max=[], solved=[], shape=set()) for mode in MODES}
        for k, (q, lo, hi) in enumerate(seq):
            for mode in MODES[k % 4:] + MODES[:k % 4]:
                h.upload(q, lo, hi)
                if mode != "cold":
                    xp, yp = prev[mode]
                    h.warm_start(xp if "x" in mode else None, yp if "y" in mode else None)
                ms = h.solve_resident(nb)
                x, y, infos = h.download(nb)
                it = np.array([i["iter"] for i in infos])
                r = rec[mode]
                r["ms"].append(ms)
                r["iter_mean"].append(float(it.mean()))
                r["iter_max"].append(int(it.max()))
                r["solved"].append(sum(i["status_val"] == 1 for i in infos))
                r["shape"].add(h.last_shape())
                prev[mode] = (x, y)
    finally:
        h.cleanup()
    out = {}
    for mode, r in rec.items():
        out[mode] = dict(ms_per_step_mean=float(np.mean(r["ms"])), ms_per_step=[round(v, 3) for v in r["ms"]],
                         iter_mean=float(np.mean(r["iter_mean"])), iter_max=max(r["iter_max"]),
                         iter_max_per_step=r["iter_max"], solved=int(sum(r["solved"])), solves=nb * len(seq),
                         shape=sorted(r["shape"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--nb", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--drifts", default="0.001,0.01")
    ap.add_argument("--seed", type=int, default=0)
    a = ap.parse_args()
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, nb=a.nb, n=240, m=949, steps=a.steps, seed=a.seed,
               timing="device ms of solve_resident (solve kernels only) per step; modes alternate within each step",
               drifts={})
    for d in (float(s) for s in a.drifts.split(",")):
        res["drifts"][str(d)] = run_drift(a.nb, a.steps, d, a.seed)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "batch_warm.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    for d, modes in res["drifts"].items():
        for mode, r in modes.items():
            print(f"drift {d:>6} {mode:>4}: {r['ms_per_step_mean']:8.2f} ms/step  iter mean {r['iter_mean']:6.1f} max {r['iter_max']:4d}  "
                  f"solved {r['solved']}/{r['solves']}  shape {r['shape']}")


if __name__ == "__main__":
    main()
