"""Host-side checks of the radial export (dftatom_solve_batch_radial): the build, the ctypes mirror of dftatom_radial, the orbital-row
count the Python layer sizes its arrays with, and the CLI flag.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import pytest

import dftatom_b200 as D
import oracle_lib as O
from dftatom_b200.api import _CRadial

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_holds_the_export_kernels_for_sm_100a():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    D.load_library()
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "radial_orbitals_kernel" in out and "radial_fields_kernel" in out
    lib = D.load_library()
    assert hasattr(lib, "dftatom_solve_batch_radial") and hasattr(lib, "dftatom_radial_moments")


def test_ctypes_radial_matches_the_c_layout():
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in _CRadial._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += '    printf("%zu %d\\n", sizeof(dftatom_radial), DFTATOM_N_MOMENTS);\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof(dftatom_radial, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()
    assert int(vals[0]) == C.sizeof(_CRadial)
    assert int(vals[1]) == D.api.N_MOMENTS
    assert [int(v) for v in vals[2:]] == [getattr(_CRadial, f).offset for f in fields]


def test_orbital_count_equals_the_levels_of_every_atom():
    for Z in range(1, 119):
        assert D.orbital_count(Z, 0) == len(O.aufbau(Z)) == len(D.aufbau(Z))
        oa, ob, _, _ = O.split_spin(Z)
        a, b, _, _ = D.split_spin(Z)
        assert D.orbital_count(Z, 1) == len(oa) + len(ob) == len(a) + len(b)
        assert D.orbital_count(Z, 2) == D.orbital_count(Z, 0) and D.orbital_count(Z, 3) == D.orbital_count(Z, 1)


def test_cli_help_names_the_radial_flag():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--radial DIR" in out
