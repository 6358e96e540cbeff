"""Profiling driver for the dense Newton kernels (run under ncu): one blocked Cholesky, one SYRK, one updown sweep."""
import ctypes as C
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from qpalm_b200.interface import load_library
from qpalm_b200 import abi
n = int(sys.argv[1]) if len(sys.argv) > 1 else 8000
what = sys.argv[2] if len(sys.argv) > 2 else "potrf"
lib = load_library("b200")
ms = C.c_double(0)
if what == "potrf":
    lib.qpalm_b200_bench_potrf.argtypes = [abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    rc = lib.qpalm_b200_bench_potrf(n, 1, C.byref(ms))
    print("potrf", n, "rc", rc, "ms", ms.value, "TFLOP/s", n**3 / 3 / ms.value / 1e9)
elif what == "syrk":
    k = int(sys.argv[3]) if len(sys.argv) > 3 else 4000
    lib.qpalm_b200_bench_dsyrk.argtypes = [abi.c_int, abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    rc = lib.qpalm_b200_bench_dsyrk(n, k, 2, C.byref(ms))
    print("syrk", n, k, "ms", ms.value, "TFLOP/s", n * n * k / ms.value / 1e9)
elif what == "updown":
    lib.qpalm_b200_bench_updown.argtypes = [abi.c_int, abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    for k in ([int(sys.argv[3])] if len(sys.argv) > 3 else [1, 8, 32, 33, 64]):
        rc = lib.qpalm_b200_bench_updown(n, k, 3, C.byref(ms))
        npad = (n + 127) // 128 * 128
        print("updown sweep n", n, "k", k, "rc", rc, "ms", round(ms.value, 4), "us per 32-column panel", round(1e3 * ms.value / (npad / 32), 3),
              "GB/s (2 B_L)", round(2 * 8 * npad * (npad + 1) / 2 / ms.value / 1e6, 1))
elif what == "potrf_prof":
    # per-kernel CUDA-event breakdown of one blocked Cholesky
    lib.qpalm_b200_bench_potrf.argtypes = [abi.c_int, abi.c_int, C.POINTER(C.c_double)]
    lib.qpalm_b200_bench_potrf(n, 1, C.byref(ms))
    lib.qpalm_b200_prof_enable(b"*")
    lib.qpalm_b200_bench_potrf(n, 0, C.byref(ms))
    buf = C.create_string_buffer(1 << 16)
    lib.qpalm_b200_prof_report(buf, len(buf))
    import json
    rep = json.loads(buf.value.decode())
    for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"]):
        print(f"  {k:28s} launches {v['launches']:6d}  ms {v['ms']:9.3f}  mean_us {1e3 * v['ms'] / v['launches']:8.2f}")
