"""Host-side checks of the self-consistent pseudo-atom (dftatom_solve_pseudo_batch): the ctypes mirror of dftatom_pseudo_atom, the
entry and its kernel in the library, the CLI flag --pseudo-test and its errors, and a CPU self-check of the reference of
tests/pseudo_scf_ref.py: carbon solved by the CPU oracle, pseudized by tests/pseudo_ref.py and re-solved as a pseudo-atom in its reference
configuration reproduces the all-electron valence eigenvalues.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import oracle_config_lib as OC
import oracle_lib as O
import pseudo_ref as P
import pseudo_scf_ref as PS
from dftatom_b200.api import _CPseudoAtom

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_struct_matches_the_c_layout():
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in _CPseudoAtom._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += '    printf("%zu\\n", sizeof(dftatom_pseudo_atom));\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof(dftatom_pseudo_atom, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == C.sizeof(_CPseudoAtom) == 56
    assert vals[1:] == [getattr(_CPseudoAtom, f).offset for f in fields]


def test_library_exports_the_entry_and_holds_the_kernel_for_sm_100a():
    lib = D.load_library()
    assert hasattr(lib, "dftatom_solve_pseudo_batch")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "pseudo_potential_energy_kernel" in out


def test_cli_help_names_the_flag_and_rejects_bad_uses():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--pseudo-test" in out
    with tempfile.TemporaryDirectory() as tmp:
        ps = ["--pseudo", os.path.join(tmp, "ps"), "--pseudo-rc", "2"]
        # refused before any device work: without --pseudo, with several atoms, an unreadable configuration
        for extra in (["--Z", "14", "--pseudo-test", "3s1 3p3"], ["--Z", "6,14"] + ps + ["--pseudo-test", "3s1 3p3"],
                      ["--Z", "14"] + ps + ["--pseudo-test", "3s1 3q3"], ["--Z", "14"] + ps + ["--pseudo-test", "3s1 3p3;;"]):
            p = subprocess.run([exe] + extra, capture_output=True, text=True)
            assert p.returncode == 2, (extra, p.stderr)


GRID = (12, 0.002, 25.0)          # 4097 nodes: the radii of the GPU tests' 16385-node grid (same Rp)


@pytest.fixture(scope="module")
def carbon():
    levels, delta, max_r = GRID
    cfg = [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, 2.0)]
    ae = OC.scf_config(6, levels, 0.5, max_r, delta, 0, cfg, export=True)
    assert ae["finished"]
    V = ae["V"][0]
    eps = ae["steps"][-1]["E"][0]            # (n, l) order: 1s 2s 2p
    chans = []
    for k, l in ((1, 0), (2, 1)):
        u, _ = O.orbital(V, delta, max_r, l, eps[k])
        chans.append((P.tm_channel(V, u, levels, delta, max_r, l, eps[k], 1.5), l, 2.0))
    _, _, _, vion = P.unscreen(levels, delta, max_r, chans)
    assert all(ch["status"] == 0 for ch, _, _ in chans)
    return dict(eps=eps, v_ion={0: vion[0], 1: vion[1]}, chans=chans)


def test_reference_pseudo_atom_reproduces_the_all_electron_valence_levels(carbon):
    levels, delta, max_r = GRID
    ps = PS.solve(carbon["v_ion"], {0: 2, 1: 2}, [(2, 0, 0, 2.0), (2, 1, 0, 2.0)], levels, delta, max_r)
    assert ps["converged"]
    # self-consistency of the all-electron atom and of the pseudo-atom: both stop at |dE/E| < 1e-11
    assert abs(ps["E"][0][0] - carbon["eps"][1]) < 2e-6, (ps["E"], carbon["eps"])
    assert abs(ps["E"][0][1] - carbon["eps"][2]) < 2e-6, (ps["E"], carbon["eps"])
    # the reported energies add up at convergence (definition in include/dftatom_b200.h)
    assert abs(ps["Ekin"] + ps["Eenuc"] + ps["Ecoul"] + ps["Exc"] - ps["Etotal"]) < 1e-8
    assert ps["Ekin"] > 0 and ps["Ecoul"] > 0 and ps["Eenuc"] < 0


def test_z_bracket_keeps_a_10_hartree_margin():
    assert PS.z_bracket([np.array([0.0, -5.0, -1.0])]) == 4          # -17 <= -15
    assert PS.z_bracket([np.array([0.0, 3.0]), np.array([0.0, 8.0])]) == 3          # -10 <= -7
