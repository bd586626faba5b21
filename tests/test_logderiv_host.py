"""Host-side checks of the logarithmic derivatives (dftatom_log_derivatives): the ctypes mirror of dftatom_logderiv, the kernel in the
library, the CLI flags, and the numpy reference against the hydrogen atom.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import logderiv_ref as R
from dftatom_b200.api import _CLogDeriv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_logderiv_matches_the_c_layout():
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in _CLogDeriv._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += '    printf("%zu\\n", sizeof(dftatom_logderiv));\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof(dftatom_logderiv, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == C.sizeof(_CLogDeriv) == 32
    assert vals[1:] == [getattr(_CLogDeriv, f).offset for f in fields]


def test_library_exports_the_entry_and_holds_the_kernel_for_sm_100a():
    lib = D.load_library()
    assert hasattr(lib, "dftatom_log_derivatives")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out and "logderiv_kernel" in out


def test_cli_help_names_the_logderiv_flags():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--logderiv DIR" in out and "--rc R" in out and "--energies lo:hi:n" in out


def _hydrogen(levels, delta):
    N, r, _, _ = R.grid(levels, delta, 25.0)
    V = np.zeros(N)
    V[1:] = -1.0 / r[1:]
    return V


@pytest.mark.parametrize("levels,delta,tol", [(12, 0.002, 1e-8), (14, 0.0005, 1e-10)])
def test_reference_meets_hydrogen(levels, delta, tol):
    V = _hydrogen(levels, delta)
    D0, u0, _, n0, rc = R.log_derivative(V, levels, delta, 25.0, 0, 2.0, [-0.5])
    D1, u1, _, n1, _ = R.log_derivative(V, levels, delta, 25.0, 1, 2.0, [-0.125])
    assert abs(rc - 2.0) < 0.01
    assert abs(D0[0] - (1 / rc - 1)) < tol and abs(D1[0] - (2 / rc - 0.5)) < tol
    # u = r e^-r (1s), r^2 e^(-r/2) (2p), normalised on [0, r_c]
    i0 = 0.25 - np.exp(-2 * rc) * (rc * rc / 2 + rc / 2 + 0.25)
    i1 = 24 - np.exp(-rc) * (rc ** 4 + 4 * rc ** 3 + 12 * rc ** 2 + 24 * rc + 24)
    assert abs(u0[0] - rc * np.exp(-rc) / np.sqrt(i0)) < tol and abs(u1[0] - rc * rc * np.exp(-rc / 2) / np.sqrt(i1)) < tol
    assert n0[0] == 0 and n1[0] == 0


def test_reference_phase_is_monotone_and_wronskian_holds():
    V = _hydrogen(12, 0.002)
    E = np.linspace(-3.0, 5.0, 4001)
    for l in range(4):
        Dv, u, _, nodes, rc = R.log_derivative(V, 12, 0.002, 25.0, l, 2.0, E)
        assert np.all(nodes >= 0) and np.all(np.diff(R.phase(Dv, nodes, rc)) > 0)
    E = np.linspace(-3.0, 5.0, 201)
    h = 1e-5
    for l in range(4):
        Dv, u, _, _, rc = R.log_derivative(V, 12, 0.002, 25.0, l, 2.0, E)
        dD = (R.log_derivative(V, 12, 0.002, 25.0, l, 2.0, E + h)[0] - R.log_derivative(V, 12, 0.002, 25.0, l, 2.0, E - h)[0]) / (2 * h)
        ok = np.abs(rc * Dv) < 20
        assert ok.sum() > 100
        assert np.max(np.abs(-0.5 * dD[ok] * u[ok] ** 2 - 1)) < 1e-5


def test_reference_flags_a_coarse_grid_and_stays_finite_deep_down():
    # uniform grid of 257 nodes (h = 0.098), E far below the potential: g = h^2 (V - E) / 6 > 1
    N, r, _, _ = R.grid(8, 0.0, 25.0)
    V = np.zeros(N)
    V[1:] = -1.0 / r[1:]
    Dv, u, du, nodes, _ = R.log_derivative(V, 8, 0.0, 25.0, 0, 10.0, [-2000.0, 0.5])
    assert nodes[0] == -1 and np.isnan(Dv[0]) and np.isnan(u[0]) and np.isnan(du[0])
    assert nodes[1] >= 0 and np.isfinite(Dv[1])
    # E = -Z^2 - 1 at r_(N-2): the solution grows by ~e^3000, the rescaled sweep stays finite
    N, r, _, _ = R.grid(14, 0.0005, 25.0)
    V = np.zeros(N)
    V[1:] = -86.0 / r[1:]
    out = R.log_derivative(V, 14, 0.0005, 25.0, 0, r[N - 2], [-86.0 ** 2 - 1])
    assert all(np.isfinite(x).all() for x in out[:3]) and out[3][0] == 0
