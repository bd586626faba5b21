"""TEST INFRASTRUCTURE: ctypes access to the oracle's SCF of an electron configuration (orc_scf_config, oracle/dftatom_oracle_config.c).
The library is compiled from the oracle's sources on first use into a temporary directory (the tree may be read-only where tests run)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle_lib import MAXLV, ORACLE_DIR, STEP_CB, OrcOptions, OrcResult, d

_dp = C.POINTER(C.c_double)


class OrcOrbital(C.Structure):
    _fields_ = [("n", C.c_int), ("l", C.c_int), ("spin", C.c_int), ("occ", C.c_double)]


class OrcConfig(C.Structure):
    _fields_ = [("n_orbitals", C.c_int), ("orb", OrcOrbital * (2 * MAXLV))]


_lib = None


def oracle_config():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="dftatom_oracle_config_")
        atexit.register(shutil.rmtree, tmp, True)
        path = os.path.join(tmp, "libdftatom_oracle_config.so")
        cc = shutil.which("cc") or shutil.which("gcc") or "gcc"
        # -Bsymbolic: the orc_* functions this library carries bind to its own copies, not to libdftatom_oracle.so's
        subprocess.run([cc, "-std=c11", "-O2", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-o", path, os.path.join(ORACLE_DIR, "dftatom_oracle_config.c"),
                        "-lm"], check=True)
        L = C.CDLL(path)
        L.orc_scf_config.argtypes = [C.POINTER(OrcOptions), C.POINTER(OrcConfig), C.POINTER(OrcResult), STEP_CB, C.c_void_p, C.c_int, _dp, _dp]
        _lib = L
    return _lib


def scf_config(Z, levels, mixing, max_r, delta, method, config, max_vcycles=100, export=False):
    """The oracle SCF of a configuration: a list of (n, l, spin, occ) entries.  Returns the dict of oracle_lib.scf (the records' occ is
    rounded); export=True adds V and rho, [2][N] each (the arrays of orc_scf_ex)."""
    steps = []

    def cb(st, _):
        s = st.contents
        steps.append(dict(step=s.step,
                          E=[[s.lv[sp][k].E for k in range(s.n_levels[sp])] for sp in range(2)],
                          levels=[[(s.lv[sp][k].n0 + 1, s.lv[sp][k].l, s.lv[sp][k].occ) for k in range(s.n_levels[sp])] for sp in range(2)],
                          Etotal=s.Etotal, Ekin=s.Ekin, Ecoul=s.Ecoul, Eenuc=s.Eenuc, Exc=s.Exc, ok=s.level_search_converged))

    o = OrcOptions(Z, levels, max_r, delta, mixing, method)
    r = OrcResult()
    cfg = OrcConfig()
    cfg.n_orbitals = len(config)
    for k, (n, l, spin, occ) in enumerate(config):
        cfg.orb[k] = OrcOrbital(int(n), int(l), int(spin), float(occ))
    N = 2 ** int(levels) + 1
    V = np.zeros((2, N)) if export else None
    rho = np.zeros((2, N)) if export else None
    rc = oracle_config().orc_scf_config(C.byref(o), C.byref(cfg), C.byref(r), STEP_CB(cb), None, max_vcycles, d(V) if export else None,
                                        d(rho) if export else None)
    if rc != 0:
        raise ValueError(f"orc_scf_config rejected the configuration {config}")
    nsp = 2 if method in (1, 3) else 1
    out = dict(steps=steps, finished=bool(r.finished), n_steps=r.n_steps,
               sorted=[[(r.sorted[sp][k].n0 + 1, r.sorted[sp][k].l, r.sorted[sp][k].occ) for k in range(r.n_sorted[sp])] for sp in range(nsp)])
    if export:
        out.update(V=V, rho=rho)
    return out
