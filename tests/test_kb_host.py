"""Host-side checks of the Kleinman-Bylander calls (dftatom_kb_form, dftatom_kb_log_derivatives): the ctypes mirrors of their structs,
the kernels in the library, the CLI flag, and the numpy reference of tests/kb_ref.py on smooth model potentials.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.special import erf

import dftatom_b200 as D
import kb_ref as K
import logderiv_ref as LR
from dftatom_b200.api import _CKbChannel, _CKbLdChannel, _CKbResult

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("cls,name,size", [(_CKbChannel, "dftatom_kb_channel", 24), (_CKbResult, "dftatom_kb_result", 56),
                                           (_CKbLdChannel, "dftatom_kb_ld_channel", 32)])
def test_ctypes_structs_match_the_c_layout(cls, name, size):
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in cls._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += f'    printf("%zu\\n", sizeof({name}));\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof({name}, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == C.sizeof(cls) == size
    assert vals[1:] == [getattr(cls, f).offset for f in fields]


def test_library_exports_the_entries_and_holds_the_kernels_for_sm_100a():
    lib = D.load_library()
    assert hasattr(lib, "dftatom_kb_form") and hasattr(lib, "dftatom_kb_log_derivatives")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    for k in ("kb_form_kernel", "kb_proj_kernel", "kb_logderiv_kernel"):
        assert k in out


def test_cli_help_names_the_flag_and_rejects_bad_uses():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--pseudo-local L" in out
    with tempfile.TemporaryDirectory() as tmp:
        # refused before any device work: without --pseudo, and an l outside 0..3
        for extra in (["--pseudo-local", "1"], ["--pseudo", os.path.join(tmp, "ps"), "--pseudo-rc", "2", "--pseudo-local", "4"],
                      ["--pseudo", os.path.join(tmp, "ps"), "--pseudo-rc", "2", "--pseudo-local", "p"]):
            p = subprocess.run([exe, "--Z", "14"] + extra, capture_output=True, text=True)
            assert p.returncode == 2, (extra, p.stderr)


GRID = (11, 0.005, 20.0)


def _model(A, l=0, rs=1.5):
    """A Gaussian-screened Coulomb well V_row = -3 erf(r) / r, its nodeless level eps and orbital (the reference's own), and the local
    potential V_row - A (1 - (r/rs)^2)^3 inside rs (equal to V_row beyond rs)."""
    N, r, _, _ = LR.grid(*GRID)
    rr = np.where(r > 0, r, 1.0)
    V = np.where(r > 0, -3.0 * erf(rr) / rr, 0.0)
    Vloc = V - A * np.where(r < rs, (1 - (r / rs) ** 2) ** 3, 0.0)
    eps = K.local_levels(V, *GRID, l, k=1)[0]
    n = LR.nearest_node(r, 4.0)
    u = np.zeros(N)
    u[:n + 1] = K.outward(V, *GRID, l, eps, n) * np.exp(0.5 * GRID[1] * np.arange(n + 1))
    return np.stack([V, Vloc]), np.stack([u, u]), eps


@pytest.mark.parametrize("A", [-1.0, 10.0])
def test_kb_log_derivative_at_the_reference_energy_equals_the_semilocal_one(A):
    V, u, eps = _model(A)
    kb = K.kb_form(V, u, *GRID, 0, 1, 0, eps)
    assert kb["status"] == 0 and abs(np.sum(LR.simpson_weights(kb["i_s"]) * kb["beta"][:kb["i_s"] + 1] ** 2 *
                                            LR.grid(*GRID)[3][:kb["i_s"] + 1]) - 1) < 1e-12
    D_kb, u_kb, du_kb, n_kb, _ = K.kb_log_derivative(V[1], kb["beta"], *GRID, 0, kb["E_KB"], 2.0, [eps])
    D_sl, u_sl, du_sl, n_sl, _ = LR.log_derivative(V[0], *GRID, 0, 2.0, [eps])
    # the KB term reproduces dV u exactly at eps on the nodes, and its Numerov source is weighted like the potential's: rounding only
    assert abs(D_kb[0] - D_sl[0]) < 1e-9 * abs(D_sl[0]) and abs(u_kb[0] - u_sl[0]) < 1e-9 * abs(u_sl[0]) and n_kb[0] == n_sl[0]


@pytest.mark.parametrize("A,ghost", [(10.0, 0), (30.0, 1)])
def test_gss_verdict_equals_the_dense_check(A, ghost):
    V, u, eps = _model(A)
    kb = K.kb_form(V, u, *GRID, 0, 1, 0, eps)
    eps_loc = K.local_levels(V[1], *GRID, 0)
    assert kb["E_KB"] > 0
    assert K.gss_ghost(kb["E_KB"], eps, eps_loc) == ghost
    assert K.dense_ghost(V[1], kb["beta"], *GRID, 0, kb["E_KB"], eps, margin=1e-3, coarse_levels=GRID[0]) == ghost
