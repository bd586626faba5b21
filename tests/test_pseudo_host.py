"""Host-side checks of the Troullier-Martins pseudization (dftatom_tm_pseudize): the ctypes mirrors of dftatom_tm_channel and
dftatom_tm_result, the kernels in the library, and the numpy reference of tests/pseudo_ref.py on hydrogen 2s / 2p.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.integrate import quad
from scipy.optimize import brentq

import dftatom_b200 as D
import logderiv_ref as LR
import pseudo_ref as P
from dftatom_b200.api import _CTmChannel, _CTmResult

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("cls,name,size", [(_CTmChannel, "dftatom_tm_channel", 40), (_CTmResult, "dftatom_tm_result", 80)])
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


def test_library_exports_the_entry_and_holds_the_kernels_for_sm_100a():
    lib = D.load_library()
    assert hasattr(lib, "dftatom_tm_pseudize")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    for k in ("tm_kernel", "tm_density_kernel", "tm_unscreen_kernel"):
        assert k in out


def _hydrogen(levels, delta, max_r=25.0):
    N, r, _, jac = LR.grid(levels, delta, max_r)
    V = np.zeros(N)
    V[1:] = -1.0 / r[1:]
    return V, r, jac


# (l, u(r), r_c): hydrogen 2s (node at r = 2) and 2p, eps = -1/8
CASES = [(0, lambda r: r * (1 - r / 2) * np.exp(-r / 2), 3.0), (0, lambda r: r * (1 - r / 2) * np.exp(-r / 2), 4.0),
         (1, lambda r: r * r * np.exp(-r / 2), 1.0), (1, lambda r: r * r * np.exp(-r / 2), 2.5)]


@pytest.mark.parametrize("l,uf,r_c", CASES, ids=["2s-3", "2s-4", "2p-1", "2p-2.5"])
def test_reference_meets_the_definition_on_hydrogen(l, uf, r_c):
    levels, delta = 13, 0.001
    V, r, jac = _hydrogen(levels, delta)
    u = uf(r)
    out = P.tm_channel(V, u, levels, delta, 25.0, l, -0.125, r_c)
    assert out["status"] == 0
    c, rc, n = out["c"], out["r_c"], out["n"]
    # continuity of p .. p'''' at r_c: the polynomial's derivatives against the targets
    poly = np.polynomial.Polynomial(np.ravel(np.column_stack([c, np.zeros(7)]))[:13])
    target = out["ae"]["p"]
    for k in range(5):
        got = poly.deriv(k)(rc) if k else poly(rc)
        assert abs(got - target[k]) <= 1e-9 * max(1.0, abs(target[k])), (k, got, target[k])
    assert abs(c[1] ** 2 + (2 * l + 5) * c[2]) <= 1e-12 * c[1] ** 2
    # norm conservation on the grid, and the root the definition picks: negative x, the smaller |c2|
    S = np.sum(LR.simpson_weights(n) * out["u_ps"][:n + 1] ** 2 * jac[:n + 1])
    assert abs(S / out["q"] - 1) < 1e-12
    assert -16.5 < out["x"] < 0
    # u_ps and V_scr meet the all-electron rows at r_c and copy them beyond
    assert abs(out["u_ps"][n] - abs(u[n])) <= 1e-12 * abs(u[n])
    assert np.array_equal(out["u_ps"][n + 1:], np.sign(u[n]) * u[n + 1:]) and np.array_equal(out["v_scr"][n + 1:], V[n + 1:])
    assert abs(out["v_scr"][n] - V[n]) < 1e-9


@pytest.mark.parametrize("l,uf,r_c", CASES[::2], ids=["2s-3", "2p-1"])
def test_reference_c2_converges_to_the_continuous_norm_condition(l, uf, r_c):
    levels, delta = 15, 0.00025
    V, r, jac = _hydrogen(levels, delta)
    out = P.tm_channel(V, uf(r), levels, delta, 25.0, l, -0.125, r_c)
    ae, rc = out["ae"], out["r_c"]
    vecs = P.coeff_vectors(ae, l)
    q = quad(lambda x: uf(x) ** 2, 0, rc, epsabs=0, epsrel=1e-13, limit=200)[0]

    def F(x):
        d = P.scaled_coeffs(ae, l, x, vecs)
        S = quad(lambda t: rc * (rc * t) ** (2 * l + 2) * np.exp(2 * np.polynomial.polynomial.polyval(t * t, d)), 0, 1,
                 epsabs=0, epsrel=1e-13, limit=200)[0]
        return np.log(S) - np.log(q)
    k = int(np.floor(-2 * out["x"]))
    x_cont = brentq(F, -0.5 * (k + 1), -0.5 * k, xtol=1e-15, rtol=1e-14)
    assert abs(out["x"] - x_cont) <= 1e-6 * abs(x_cont)


def test_reference_unscreening_of_a_hydrogen_like_valence():
    levels, delta = 12, 0.002
    V, r, _ = _hydrogen(levels, delta)
    u = r * r * np.exp(-r / 2)
    ch = P.tm_channel(V, u, levels, delta, 25.0, 1, -0.125, 2.0)
    rho, vh, vxc, (vion,) = P.unscreen(levels, delta, 25.0, [(ch, 1, 1.0)])
    n = ch["n"]
    # one electron: U(R) = 1, so r V_H = 1 at the last node
    assert abs(r[-1] * vh[-1] - 1) < 1e-12
    assert np.all(np.isfinite(vion)) and vion[0] == 0.0
    assert np.allclose(vion[n + 1:], V[n + 1:] - vh[n + 1:] - vxc[n + 1:], rtol=0, atol=1e-15)
    # a failed channel makes the whole row NaN
    bad = dict(ch, status=1)
    rho, _, _, (vion,) = P.unscreen(levels, delta, 25.0, [(bad, 1, 1.0)])
    assert rho[0] == 0 and np.all(np.isnan(rho[1:])) and np.all(np.isnan(vion[1:]))


def test_cli_help_names_the_pseudo_flags_and_rejects_lsda():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--pseudo DIR" in out and "--pseudo-rc Rs[,Rp,Rd,Rf]" in out
    with tempfile.TemporaryDirectory() as tmp:
        # refused before any device work: LSDA atoms, unreadable radii, and a log-derivative radius inside a pseudo radius
        for extra in (["--method", "1", "--pseudo-rc", "2"], ["--pseudo-rc", "2,x"], ["--pseudo-rc", "2,2.5", "--logderiv", tmp, "--rc", "2.2"]):
            p = subprocess.run([exe, "--Z", "14", "--pseudo", os.path.join(tmp, "ps")] + extra, capture_output=True, text=True)
            assert p.returncode == 2, (extra, p.stderr)
