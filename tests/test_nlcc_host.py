"""Host-side checks of the nonlinear core correction (dftatom_partial_core, dftatom_tm_pseudize_core, dftatom_solve_pseudo_batch_core):
the ctypes mirrors of the new structs, the entries and kernels in the library, the CLI flag --pseudo-core and its errors, self-checks of
the reference of tests/nlcc_ref.py, and the end-to-end chain on the CPU: carbon solved by the CPU oracle, pseudized with a core and
re-solved as a core-corrected pseudo-atom reproduces the all-electron valence eigenvalues.  No GPU needed."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import logderiv_ref as LR
import nlcc_ref as NR
import oracle_config_lib as OC
import oracle_lib as O
import pseudo_ref as P
from dftatom_b200.api import _CCoreOrbital, _CPccResult

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("ctype,cname,size", [(_CCoreOrbital, "dftatom_core_orbital", 16), (_CPccResult, "dftatom_pcc_result", 56)])
def test_ctypes_structs_match_the_c_layout(ctype, cname, size):
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in ctype._fields_]
    src = "#include <stddef.h>\n#include <stdio.h>\n#include \"dftatom_b200.h\"\nint main(void) {\n"
    src += f'    printf("%zu\\n", sizeof({cname}));\n'
    for f in fields:
        src += f'    printf("%zu\\n", offsetof({cname}, {f}));\n'
    src += "    return 0;\n}\n"
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "layout.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(tmp, "layout")
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(tmp, "layout.c")], check=True)
        vals = [int(v) for v in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == C.sizeof(ctype) == size
    assert vals[1:] == [getattr(ctype, f).offset for f in fields]


def test_library_exports_the_entries_and_holds_the_kernels_for_sm_100a():
    lib = D.load_library()
    for name in ("dftatom_partial_core", "dftatom_tm_pseudize_core", "dftatom_solve_pseudo_batch_core"):
        assert hasattr(lib, name)
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-elf", D.lib_path()], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "partial_core_kernel" in out
    assert "core_xc_density_kernel" in out
    assert "pseudo_potential_energy_kernelILb1E" in out and "pseudo_potential_energy_kernelILb0E" in out


def test_cli_help_names_the_flag_and_rejects_bad_uses():
    exe = os.path.join(ROOT, "bin", "dftatom")
    if not os.path.exists(exe):
        pytest.skip("bin/dftatom not built")
    out = subprocess.run([exe, "--help"], check=True, capture_output=True, text=True).stdout
    assert "--pseudo-core" in out
    with tempfile.TemporaryDirectory() as tmp:
        ps = ["--Z", "11", "--pseudo", os.path.join(tmp, "ps"), "--pseudo-rc", "2"]
        # refused before any device work: without --pseudo, a negative, non-finite or unreadable radius
        for extra in (["--Z", "11", "--pseudo-core", "1"], ps + ["--pseudo-core", "-1"], ps + ["--pseudo-core", "nan"],
                      ps + ["--pseudo-core", "1x"], ps + ["--pseudo-core", ""]):
            p = subprocess.run([exe] + extra, capture_output=True, text=True)
            assert p.returncode == 2, (extra, p.stderr)


GRID = (12, 0.002, 25.0)          # 4097 nodes: the grid of tests/test_pseudo_scf_host.py


@pytest.fixture(scope="module")
def carbon():
    levels, delta, max_r = GRID
    cfg = [(1, 0, 0, 2.0), (2, 0, 0, 2.0), (2, 1, 0, 2.0)]
    ae = OC.scf_config(6, levels, 0.5, max_r, delta, 0, cfg, export=True)
    assert ae["finished"]
    V = ae["V"][0]
    eps = ae["steps"][-1]["E"][0]            # (n, l) order: 1s 2s 2p
    u1s, _ = O.orbital(V, delta, max_r, 0, eps[0])
    rho_core = NR.core_density([u1s], [2.0], levels, delta, max_r)
    chans = []
    for k, l in ((1, 0), (2, 1)):
        u, _ = O.orbital(V, delta, max_r, l, eps[k])
        chans.append((P.tm_channel(V, u, levels, delta, max_r, l, eps[k], 1.5), l, 2.0))
    assert all(ch["status"] == 0 for ch, _, _ in chans)
    return dict(eps=eps, rho_core=rho_core, chans=chans)


def test_reference_partial_core_matches_value_and_slope_at_r_pc(carbon):
    levels, delta, max_r = GRID
    N, r, _, _ = LR.grid(levels, delta, max_r)
    rc = carbon["rho_core"]
    # the 1s density of carbon holds its two electrons (Simpson 3/8 weights of the radial export)
    assert abs(NR.partial_core(rc, levels, delta, max_r, 0.0)["n_core"] - 2.0) < 1e-6
    for r_pc in (0.3, 0.6, 1.0):
        pc = NR.partial_core(rc, levels, delta, max_r, r_pc)
        assert pc["status"] == 0
        n, A, B = pc["i_pc"], pc["A"], pc["B"]
        x = B * pc["r_pc"]
        assert 0 < x < np.pi and abs(x * np.cos(x) - pc["t"] * np.sin(x)) < 1e-14
        # value and slope of A sin(Br) / r at r_pc equal rho_core and its derivative there
        assert abs(A * np.sin(x) / pc["r_pc"] - rc[n]) <= 1e-13 * rc[n]
        slope = A * (x * np.cos(x) - np.sin(x)) / pc["r_pc"] ** 2
        J = delta * (pc["r_pc"] + max_r / (np.exp((N - 1) * delta) - 1.0))
        d = ((rc[n - 2] - 8 * rc[n - 1]) + (8 * rc[n + 1] - rc[n + 2])) / 12 / J
        assert abs(slope - d) <= 1e-10 * abs(d)
        assert np.all(pc["rho_pc"][1:N - 1] > 0)
        assert np.array_equal(pc["rho_pc"][n:], rc[n:])
        assert np.all(pc["rho_pc"][1:n] < rc[1:n])          # the model core is smoother and smaller inside r_pc
        assert 0 < pc["n_pc"] < pc["n_core"]
    full = NR.partial_core(rc, levels, delta, max_r, 0.0)
    assert full["status"] == 0 and np.array_equal(full["rho_pc"], rc) and full["n_pc"] == full["n_core"]
    # a density that rises at r_pc has no partial core
    bad = NR.partial_core(r ** 2, levels, delta, max_r, 1.0)
    assert bad["status"] == 1 and np.isnan(bad["A"]) and np.all(np.isnan(bad["rho_pc"][1:]))


@pytest.mark.parametrize("r_pc", [0.6, 0.0])
def test_reference_core_corrected_pseudo_atom_reproduces_the_all_electron_valence_levels(carbon, r_pc):
    levels, delta, max_r = GRID
    pc = NR.partial_core(carbon["rho_core"], levels, delta, max_r, r_pc)["rho_pc"]
    _, _, _, vion = NR.unscreen_core(levels, delta, max_r, carbon["chans"], pc)
    ps = NR.solve({0: vion[0], 1: vion[1]}, {0: 2, 1: 2}, [(2, 0, 0, 2.0), (2, 1, 0, 2.0)], levels, delta, max_r, pc)
    assert ps["converged"]
    # the tolerance of the existing host self-check (tests/test_pseudo_scf_host.py)
    assert abs(ps["E"][0][0] - carbon["eps"][1]) < 2e-6, (ps["E"], carbon["eps"])
    assert abs(ps["E"][0][1] - carbon["eps"][2]) < 2e-6, (ps["E"], carbon["eps"])
    assert abs(ps["Ekin"] + ps["Eenuc"] + ps["Ecoul"] + ps["Exc"] - ps["Etotal"]) < 1e-8
    assert ps["Ekin"] > 0 and ps["Ecoul"] > 0 and ps["Eenuc"] < 0
