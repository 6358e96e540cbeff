"""CPU suite: the C-ABI library loads, exports every symbol include/qpalm_b200.h declares, and its struct layouts are the
reference's (checked by compiling the header with gcc and comparing sizeof / offsetof with the ctypes mirror).  No compute
calls are made: there is no GPU here and the product has no CPU fallback."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

from qpalm_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "qpalm_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^[ \t]*(?:const\s+)?[A-Za-z_][A-Za-z0-9_ \*]*?[\s\*]([a-z_][A-Za-z0-9_]*)\s*\([^;{]*\)\s*;", src, flags=re.M)
    return sorted(set(n for n in names if n.startswith(("qpalm_", "validate_", "update_status"))))


def test_header_declares_the_reference_api():
    names = declared_functions()
    for f in ("qpalm_set_default_settings", "qpalm_setup", "qpalm_warm_start", "qpalm_solve", "qpalm_update_settings",
              "qpalm_update_bounds", "qpalm_update_q", "qpalm_cleanup", "qpalm_b200_batch_solve", "qpalm_b200_mat_vec",
              "qpalm_b200_linesearch", "qpalm_b200_updown"):
        assert f in names, (f, names)


def test_product_library_exports_every_declared_symbol():
    assert os.path.exists(abi.PRODUCT_LIB), "libqpalm_b200.so not built: run __graft_entry__.build()"
    lib = C.CDLL(abi.PRODUCT_LIB)
    missing = [n for n in declared_functions() if not hasattr(lib, n)]
    assert not missing, missing


def test_product_has_no_cpu_fallback_symbols():
    """The product must not link or embed the oracle."""
    out = subprocess.run(["nm", "-D", abi.PRODUCT_LIB], capture_output=True, text=True).stdout
    assert "oracle_" not in out
    ldd = subprocess.run(["ldd", abi.PRODUCT_LIB], capture_output=True, text=True).stdout
    assert "liboracle" not in ldd and "libqpalm_ref" not in ldd


def test_struct_layouts_match_ctypes_mirror(tmp_path):
    structs = {"QPALMSettings": abi.QPALMSettings, "QPALMData": abi.QPALMData, "QPALMInfo": abi.QPALMInfo,
               "QPALMSolution": abi.QPALMSolution, "QPALMScaling": abi.QPALMScaling, "QPALMSolver": abi.QPALMSolver,
               "QPALMWorkspace": abi.QPALMWorkspace, "solver_sparse": abi.SolverSparse, "array_element": abi.ArrayElement,
               "QPALMB200Stats": abi.QPALMB200Stats}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
    for name, st in structs.items():
        lines.append(f'printf("{name} size %zu\\n", sizeof({name}));')
        for fname, _ in st._fields_:
            lines.append(f'printf("{name} {fname} %zu\\n", offsetof({name}, {fname}));')
    lines.append("return 0;}")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    got = {}
    for ln in out:
        if ln:
            a, b, c = ln.split()
            got[(a, b)] = int(c)
    for name, st in structs.items():
        assert got[(name, "size")] == C.sizeof(st), name
        for fname, _ in st._fields_:
            assert got[(name, fname)] == getattr(st, fname).offset, (name, fname)


def test_struct_layouts_match_reference_headers():
    """sizeof / offsetof of the public structs compiled from the reference's own headers (CHOLMOD build), stored in
    tests/golden/reference_struct_layout.json, equal ours."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_struct_layout.json")) as f:
        ref = json.load(f)
    ref.pop("note")
    ours = {"sizeof(QPALMSettings)": C.sizeof(abi.QPALMSettings), "sizeof(QPALMData)": C.sizeof(abi.QPALMData),
            "sizeof(QPALMInfo)": C.sizeof(abi.QPALMInfo), "sizeof(QPALMSolver)": C.sizeof(abi.QPALMSolver),
            "sizeof(QPALMWorkspace)": C.sizeof(abi.QPALMWorkspace),
            "offsetof(QPALMWorkspace, solver)": abi.QPALMWorkspace.solver.offset,
            "offsetof(QPALMSolver, nb_leave)": abi.QPALMSolver.nb_leave.offset, "sizeof(cholmod_sparse)": C.sizeof(abi.SolverSparse)}
    assert ref == ours


def test_default_settings_match_reference_constants():
    """include/constants.h:65-116 -- through the oracle (CPU) twin of qpalm_set_default_settings."""
    from qpalm_b200.interface import load_library
    lib = load_library("oracle")
    s = abi.QPALMSettings()
    lib.oracle_qpalm_set_default_settings(C.byref(s))
    d = abi.default_settings_py()
    for name, _ in abi.QPALMSettings._fields_:
        assert getattr(s, name) == getattr(d, name), name


def test_product_package_never_touches_the_checkers():
    """The oracle / compiled reference are test infrastructure: no module of qpalm_b200/ may import, load or name them, and a
    fresh interpreter that imports the whole product package must know only the "b200" implementation."""
    import glob
    import subprocess
    import sys
    pkg = os.path.join(abi.REPO_ROOT, "qpalm_b200")
    for f in glob.glob(os.path.join(pkg, "*.py")):
        src = open(f).read()
        for bad in ("import oracle", "from oracle", "liboracle", "libqpalm_ref", "libqpalm_qps_ref", "oracle/_ref"):
            assert bad not in src, (f, bad)
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import qpalm_b200.interface as i, qpalm_b200.qps, qpalm_b200.batch, qpalm_b200.sparse, qpalm_b200.mpc\n"
            "assert not i._CHECKERS and 'oracle' not in sys.modules and 'oracle.refbind' not in sys.modules\n"
            "try:\n    i.load_library('oracle')\nexcept RuntimeError as e:\n    print('refused:', str(e)[:40])\n" % abi.REPO_ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert out.returncode == 0 and "refused" in out.stdout, out.stderr
