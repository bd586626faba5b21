"""ctypes binding of include/dftatom_b200.h and the Python mirror of the reference's solver surface."""
import ctypes as C
import math
import os
import re
import sys
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from .report import format_report

MAX_LEVELS = 24
MAX_STEPS_LDA = 100
MAX_STEPS_LSDA = 150
N_MOMENTS = 3            # <1/r>, <r>, <r^2> of every exported orbital (DFTATOM_N_MOMENTS)

_HERE = os.path.dirname(os.path.abspath(__file__))


class DFTAtomError(RuntimeError):
    pass


def lib_path() -> str:
    return os.path.join(_HERE, "libdftatom_b200.so")


class _COptions(C.Structure):
    _fields_ = [("Z", C.c_int), ("levels", C.c_int), ("max_r", C.c_double), ("delta", C.c_double),
                ("mixing", C.c_double), ("method", C.c_int)]


class _CLevel(C.Structure):
    _fields_ = [("n", C.c_int), ("l", C.c_int), ("occ", C.c_int), ("nodes", C.c_int), ("E", C.c_double)]


class _CStep(C.Structure):
    _fields_ = [("E", (C.c_double * MAX_LEVELS) * 2), ("Etotal", C.c_double), ("Ekin", C.c_double), ("Ecoul", C.c_double),
                ("Eenuc", C.c_double), ("Exc", C.c_double), ("levels_converged", C.c_int), ("stop_criterion_met", C.c_int)]


class _CResult(C.Structure):
    _fields_ = [("status", C.c_int), ("n_steps", C.c_int), ("n_spin", C.c_int), ("n_levels", C.c_int * 2),
                ("levels", (_CLevel * MAX_LEVELS) * 2), ("sorted", (_CLevel * MAX_LEVELS) * 2),
                ("Etotal", C.c_double), ("Ekin", C.c_double), ("Ecoul", C.c_double), ("Eenuc", C.c_double), ("Exc", C.c_double)]


class _CRadial(C.Structure):
    _fields_ = [("r", C.POINTER(C.c_double)), ("rho", C.POINTER(C.c_double)), ("v", C.POINTER(C.c_double)), ("v_hartree", C.POINTER(C.c_double)),
                ("orbitals", C.POINTER(C.c_double)), ("orbital_rows", C.c_longlong), ("moments", C.POINTER(C.c_double)),
                ("atom_moments", C.POINTER(C.c_double))]


class _CLogDeriv(C.Structure):
    _fields_ = [("D", C.c_double), ("u", C.c_double), ("du", C.c_double), ("nodes", C.c_int), ("pad", C.c_int)]


class _CTmChannel(C.Structure):
    _fields_ = [("pot", C.c_int), ("orbital", C.c_int), ("l", C.c_int), ("pad", C.c_int), ("eps", C.c_double), ("occ", C.c_double),
                ("r_c", C.c_double)]


class _CTmResult(C.Structure):
    _fields_ = [("c", C.c_double * 7), ("r_c", C.c_double), ("q", C.c_double), ("status", C.c_int), ("pad", C.c_int)]


class _CKbChannel(C.Structure):
    _fields_ = [("row", C.c_int), ("loc", C.c_int), ("l", C.c_int), ("pad", C.c_int), ("eps", C.c_double)]


class _CKbResult(C.Structure):
    _fields_ = [("E_KB", C.c_double), ("cos", C.c_double), ("eps_loc", C.c_double * 2), ("r_s", C.c_double), ("i_s", C.c_int),
                ("ghost", C.c_int), ("status", C.c_int), ("pad", C.c_int)]


class _CKbLdChannel(C.Structure):
    _fields_ = [("pot", C.c_int), ("proj", C.c_int), ("l", C.c_int), ("pad", C.c_int), ("E_KB", C.c_double), ("r_c", C.c_double)]


class _CCoreOrbital(C.Structure):
    _fields_ = [("row", C.c_int), ("orbital", C.c_int), ("occ", C.c_double)]


class _CPccResult(C.Structure):
    _fields_ = [("r_pc", C.c_double), ("A", C.c_double), ("B", C.c_double), ("n_core", C.c_double), ("n_pc", C.c_double),
                ("i_pc", C.c_int), ("status", C.c_int), ("pad", C.c_int)]


class _COccupation(C.Structure):
    _fields_ = [("n", C.c_int), ("l", C.c_int), ("spin", C.c_int), ("occ", C.c_double)]


class _CConfig(C.Structure):
    _fields_ = [("n_orbitals", C.c_int), ("orb", _COccupation * (2 * MAX_LEVELS))]


class _CPseudoAtom(C.Structure):
    _fields_ = [("row", C.c_int * 4), ("n_ref", C.c_int * 4), ("z_val", C.c_double), ("mixing", C.c_double), ("method", C.c_int),
                ("pad", C.c_int)]


_RESULT_DTYPE = np.dtype(_CResult)      # numpy views of the C structs (same layout: built from the ctypes definitions)
_STEP_DTYPE = np.dtype(_CStep)
_LEVEL_IDX = np.arange(MAX_LEVELS)[None, None, :]
_SPIN_IDX = np.arange(2)[None, :, None]


class _CProfile(C.Structure):
    _fields_ = [("ms", C.c_double), ("launches", C.c_longlong), ("work", C.c_double)]


KERNEL_CLASSES = ("search", "match", "density", "poisson", "potential")

_lib = None

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def load_library():
    """Load libdftatom_b200.so (built in-tree by __graft_entry__.build() / dftatom_b200/csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise DFTAtomError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(dftatom_b200 has no CPU fallback)")
    lib = C.CDLL(path)
    lib.dftatom_last_error.restype = C.c_char_p
    lib.dftatom_version.restype = C.c_char_p
    lib.dftatom_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    lib.dftatom_destroy.argtypes = [C.c_void_p]
    lib.dftatom_destroy.restype = None
    lib.dftatom_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
    lib.dftatom_aufbau.argtypes = [C.c_int, C.POINTER(_CLevel), C.c_int]
    lib.dftatom_split_spin.argtypes = [C.c_int, C.POINTER(_CLevel), _ip, C.POINTER(_CLevel), _ip, _ip, _ip]
    lib.dftatom_n_nodes.argtypes = [C.c_int]
    lib.dftatom_estimate_cost.argtypes = [C.c_int, C.c_int]
    lib.dftatom_estimate_cost.restype = C.c_double
    lib.dftatom_partition.argtypes = [_ip, _ip, C.c_int, C.c_int, _ip]
    lib.dftatom_solve_batch.argtypes = [C.c_void_p, C.POINTER(_COptions), C.c_int, C.POINTER(_CResult), C.POINTER(_CStep), C.c_int]
    lib.dftatom_solve_batch_radial.argtypes = [C.c_void_p, C.POINTER(_COptions), C.c_int, C.POINTER(_CResult), C.POINTER(_CStep), C.c_int,
                                               C.POINTER(_CRadial)]
    lib.dftatom_config_aufbau.argtypes = [C.c_int, C.c_int, C.c_double, C.POINTER(_CConfig)]
    lib.dftatom_solve_batch_config.argtypes = [C.c_void_p, C.POINTER(_COptions), C.POINTER(_CConfig), C.c_int, C.POINTER(_CResult),
                                               C.POINTER(_CStep), C.c_int, C.POINTER(_CRadial)]
    lib.dftatom_solve_pseudo_batch.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, C.POINTER(_CPseudoAtom),
                                               C.POINTER(_CConfig), C.c_int, C.POINTER(_CResult), C.POINTER(_CStep), C.c_int, C.POINTER(_CRadial)]
    lib.dftatom_solve_pseudo_batch_core.argtypes = lib.dftatom_solve_pseudo_batch.argtypes + [_dp, C.c_int, _ip]
    lib.dftatom_radial_moments.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, _dp]
    lib.dftatom_log_derivatives.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, _ip, _ip, _dp, C.c_int, _dp, C.c_int,
                                            C.POINTER(_CLogDeriv), _dp]
    lib.dftatom_grid_nodes.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp]
    lib.dftatom_tm_pseudize.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, _dp, C.c_int, C.POINTER(_CTmChannel), C.c_int,
                                        C.POINTER(_CTmResult), _dp, _dp, _dp, _dp]
    lib.dftatom_tm_pseudize_core.argtypes = lib.dftatom_tm_pseudize.argtypes + [_dp]
    lib.dftatom_partial_core.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, C.POINTER(_CCoreOrbital), C.c_int, _dp,
                                         C.c_int, C.POINTER(_CPccResult), _dp, _dp]
    lib.dftatom_kb_form.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, _dp, C.c_int, C.POINTER(_CKbChannel), C.c_int,
                                    C.POINTER(_CKbResult), _dp]
    lib.dftatom_kb_log_derivatives.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, _dp, C.c_int, C.POINTER(_CKbLdChannel),
                                               C.c_int, _dp, C.c_int, C.POINTER(_CLogDeriv), _dp]
    lib.dftatom_last_timing.argtypes = [C.c_void_p, _dp, C.POINTER(C.c_longlong)]
    lib.dftatom_last_graph_iterations.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
    lib.dftatom_last_transfer.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    lib.dftatom_last_profile.argtypes = [C.c_void_p, C.POINTER(_CProfile)]
    lib.dftatom_measure_fp64_peak.argtypes = [C.c_void_p, _dp]
    lib.dftatom_numerov_lanes.argtypes = [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_int, _ip, _dp, _ip, C.c_int, _ip, _dp, _ip]
    lib.dftatom_numerov_lanes_timed.argtypes = [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_int, _ip, _dp, _ip, C.c_int, _ip, _dp, _ip,
                                                C.c_int, C.POINTER(C.c_float), _dp]
    lib.dftatom_level_search.argtypes = [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, _ip, _ip, _dp, _ip]
    lib.dftatom_numerov_orbital.argtypes = [C.c_void_p, _dp, C.c_int, C.c_double, C.c_double, C.c_int, C.c_double, _dp, _ip]
    lib.dftatom_poisson_solve.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, _ip, _dp, _dp, _ip]
    lib.dftatom_poisson_increment.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, _dp, _dp, _dp, _ip, C.c_int, C.c_int]
    lib.dftatom_poisson_vcycles.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, _dp, _dp, C.c_int, _dp]
    lib.dftatom_vwn.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp]
    lib.dftatom_simpson38.argtypes = [C.c_void_p, C.c_double, _dp, C.c_int, C.c_int, _dp]
    lib.dftatom_xc_lda.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp]
    lib.dftatom_integrate.argtypes = [C.c_void_p, C.c_int, C.c_double, _dp, C.c_int, C.c_int, _dp]
    lib.dftatom_poisson_scratch_bytes.argtypes = [C.c_int, C.c_int]
    lib.dftatom_poisson_scratch_bytes.restype = C.c_longlong
    lib.dftatom_poisson_vcycles_dev.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p,
                                                C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_longlong)]
    _lib = lib
    return lib


def _check(rc):
    if rc < 0:
        raise DFTAtomError(f"dftatom_b200 error {rc}: {load_library().dftatom_last_error().decode()}")
    return rc


def _d(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


# ------------------------------------------------------------------------------------------------------
# data classes mirroring the reference's Options (Options.h:48-54, defaults Options.cpp:6) and Subshell
# ------------------------------------------------------------------------------------------------------
@dataclass
class Options:
    Z: int = 36
    MultigridLevels: int = 12
    MaxR: float = 10.0
    deltaGrid: float = 0.001
    alpha: float = 0.5
    method: int = 0          # 0 = LDA ("LSD" in the banner), 1 = LSDA; 2 / 3 = the same on the uniform grid (CalculateUniformLDA / LSDA)
    # beyond the reference: an ion of the reference's configuration (config_aufbau; fractional allowed, < 0 = anion), or an explicit
    # configuration - a list of (n, l, occ) (LDA) / (n, l, spin, occ) (LSDA) entries or a string for parse_config.  At most one of the two.
    charge: float = 0.0
    config: object = None

    def _c(self):
        return _COptions(int(self.Z), int(self.MultigridLevels), float(self.MaxR), float(self.deltaGrid), float(self.alpha), int(self.method))

    @property
    def configured(self) -> bool:
        return self.config is not None or float(self.charge) != 0.0

    def entries(self):
        """The configuration the atom is solved with as (n, l, spin, occ) entries, or None for the reference's Aufbau atom."""
        if self.config is not None and float(self.charge) != 0.0:
            raise DFTAtomError(f"Options(Z={self.Z}): set either `charge` or `config`, not both")
        if self.config is not None:
            cfg = parse_config(self.config, self.method) if isinstance(self.config, str) else self.config
            return [_entry4(e, self.method) for e in cfg]
        if float(self.charge) != 0.0:
            return [_entry4(e, self.method) for e in config_aufbau(self.Z, self.method, self.charge)]
        return None


@dataclass
class Level:
    n: int
    l: int
    occ: int                 # a float for an atom solved with a configuration (Options.charge / config)
    nodes: int
    E: float = 0.0


@dataclass
class Step:
    E: List[List[float]]
    Etotal: float
    Ekin: float
    Ecoul: float
    Eenuc: float
    Exc: float
    levels_converged: bool
    stop_criterion_met: bool = False


class Result:
    """One atom of a solve_batch call.  `levels` ([spin][level] in (n, l) order, eigenvalues of the last step) and `sorted_levels` (sorted by
    eigenvalue: the reference's last line) are lists of Level objects, built on first use from the (n, l, occ, nodes, E) records the library
    returned (a sweep that only reads the energies does not pay for 2000 Python objects)."""
    __slots__ = ("options", "status", "n_steps", "Etotal", "Ekin", "Ecoul", "Eenuc", "Exc", "steps", "_lv", "_sl", "radial")

    def __init__(self, options, status, n_steps, levels, sorted_levels, Etotal, Ekin, Ecoul, Eenuc, Exc, steps=None):
        self.options, self.status, self.n_steps = options, status, n_steps
        self._lv, self._sl = levels, sorted_levels            # [spin][k]: Level objects or raw tuples
        self.Etotal, self.Ekin, self.Ecoul, self.Eenuc, self.Exc = Etotal, Ekin, Ecoul, Eenuc, Exc
        self.steps = steps if steps is not None else []
        self.radial = None                 # a Radial when solve_batch(..., radial=True)

    @staticmethod
    def _as_levels(chans):
        if any(ch and not isinstance(ch[0], Level) for ch in chans):
            return [[x if isinstance(x, Level) else Level(*x) for x in ch] for ch in chans]
        return chans

    @property
    def levels(self) -> List[List[Level]]:
        self._lv = self._as_levels(self._lv)
        return self._lv

    @property
    def sorted_levels(self) -> List[List[Level]]:
        self._sl = self._as_levels(self._sl)
        return self._sl

    def __repr__(self):
        return f"Result(Z={self.options.Z}, status={self.status}, n_steps={self.n_steps}, Etotal={self.Etotal!r})"

    @property
    def finished(self) -> bool:
        return self.status == 0

    def report(self, precision: int = 6) -> str:
        """The text the reference prints for this run (DFTAtom.cpp:358-490 / :857-1021)."""
        st = []
        for s in self.steps:
            lv = []
            for sp, chan in enumerate(self.levels):
                lv += [(L.n, L.l, s.E[sp][k], L.nodes) for k, L in enumerate(chan)]
            st.append(dict(levels=lv, Etotal=s.Etotal, Ekin=s.Ekin, Ecoul=s.Ecoul, Eenuc=s.Eenuc, Exc=s.Exc))
        conf = [[(L.n, L.l, L.occ) for L in chan] for chan in self.sorted_levels]
        return format_report(self.options.Z, self.options.method, st, self.finished, conf[0], conf[1] if len(conf) > 1 else None,
                             precision, n_alpha=len(self.levels[0]))


@dataclass
class Radial:
    """The converged radial state of one atom (Context.solve_batch(..., radial=True); conventions: dftatom_solve_batch_radial in
    include/dftatom_b200.h).  Arrays are views of one allocation per batch.

    r: [N] grid nodes.  rho, V: [n_spin][N] density and Kohn-Sham potential per spin (LDA: one row, the total density).  V_H: [N]
    Hartree potential U / r.  orbitals: one [n_levels][N] array of u_nl(r) = r R_nl(r) per spin, rows aligned with Result.levels.
    moments: the same shape with N_MOMENTS columns: <1/r>, <r>, <r^2>.  n_electrons: integral of 4 pi r^2 rho.  r2: <r^2> of the
    total density summed over the electrons."""
    r: np.ndarray
    rho: np.ndarray
    V: np.ndarray
    V_H: np.ndarray
    orbitals: List[np.ndarray]
    moments: List[np.ndarray]
    n_electrons: float
    r2: float


@dataclass
class LogDerivatives:
    """Logarithmic derivatives of the outward radial solution (Context.log_derivatives; definition: dftatom_log_derivatives in
    include/dftatom_b200.h).  D, u, du, nodes: [n_channels][n_energies]; D = u'(r_c) / u(r_c) in bohr^-1, u and du the value and slope
    at r_c of the solution normalised to int_0^rc u^2 dr = 1; nodes = -1 (and NaN in D, u, du) where the grid is too coarse for the
    energy.  r_c: [n_channels] the radii actually used (nearest grid node).  E: [n_energies]."""
    D: np.ndarray
    u: np.ndarray
    du: np.ndarray
    nodes: np.ndarray
    r_c: np.ndarray
    E: np.ndarray

    @property
    def phase(self) -> np.ndarray:
        """pi nodes - atan(r_c D): continuous across the poles of D and increasing in E; NaN where nodes = -1."""
        with np.errstate(invalid="ignore"):
            ph = np.pi * self.nodes - np.arctan(self.r_c[:, None] * self.D)
        return np.where(self.nodes < 0, np.nan, ph)


@dataclass
class Pseudopotential:
    """Troullier-Martins pseudopotentials (Context.tm_pseudize / Context.pseudize; definition: dftatom_tm_pseudize in include/dftatom_b200.h).
    Per channel ([n_channels]): l, eps, occ, r_c (the radius actually used, a grid node), coefficients [n_channels][7] (c0, c2, ..., c12 of
    p(r), bohr^-2k), q (all-electron norm inside r_c), status (0 ok, 1 no root on the ladder, 2 the sweep at eps failed, 3 the root
    not refined to 1e-13), u (pseudo-orbital),
    V_scr (screened potential) and V_ion (ionic potential), each [n_channels][N].  pot: the potential row of every channel; rho_val:
    [n_pot][N] the valence density of each row.  r: [N] the grid.  n: [n_channels] the all-electron principal number of every channel's
    reference state (None when not given), which Context.solve_pseudo_batch needs."""
    l: np.ndarray
    eps: np.ndarray
    occ: np.ndarray
    r_c: np.ndarray
    coefficients: np.ndarray
    q: np.ndarray
    status: np.ndarray
    r: np.ndarray
    u: np.ndarray
    V_scr: np.ndarray
    V_ion: np.ndarray
    rho_val: np.ndarray
    pot: np.ndarray
    grid: Optional[tuple] = None        # (levels, delta, max_r) of the call, delta = 0: the uniform grid
    n: Optional[np.ndarray] = None
    rho_core: Optional[np.ndarray] = None   # [n_pot][N] core density (Context.pseudize with r_pc)
    rho_pc: Optional[np.ndarray] = None     # [n_pot][N] partial core the unscreening used; solve_pseudo_batch solves with it
    core: Optional["PartialCore"] = None    # the partial core's parameters (Context.pseudize with r_pc)


@dataclass
class PartialCore:
    """Core densities and their Louie-Froyen-Cohen partial cores (Context.partial_core; definition: dftatom_partial_core in
    include/dftatom_b200.h).  Per row ([n_rows]): r_pc (the node radius used, 0 = full core), i_pc, A, B (rho_pc = A sin(B r) / r inside
    r_pc), n_core, n_pc (electrons in rho_core / rho_pc), status (0 ok, 1 the core density does not decrease at r_pc: NaN rows);
    rho_core, rho_pc: [n_rows][N]; r: [N] the grid."""
    r_pc: np.ndarray
    i_pc: np.ndarray
    A: np.ndarray
    B: np.ndarray
    n_core: np.ndarray
    n_pc: np.ndarray
    status: np.ndarray
    rho_core: np.ndarray
    rho_pc: np.ndarray
    r: np.ndarray


@dataclass
class KleinmanBylander:
    """Kleinman-Bylander form of semilocal pseudopotentials (Context.kb_form / Context.kleinman_bylander; definition: dftatom_kb_form in
    include/dftatom_b200.h).  Per channel ([n_channels]): l, row (its potential / orbital row), loc (the row of its local potential), eps
    (reference eigenvalue), E_KB (Hartree), cos (KB cosine), eps_loc [n_channels][2] (the local Hamiltonian's eigenvalues with 0 and 1
    nodes), r_s / i_s (outermost node where V[row] != V[loc]), ghost (GSS verdict: 1 ghost below eps, 0 none, -1 undecided), status
    (0 ok, 1 local channel, 2 no projector, 3 the local search did not converge); beta: [n_channels][N] projectors; r: [N] the grid."""
    l: np.ndarray
    loc: np.ndarray
    E_KB: np.ndarray
    cos: np.ndarray
    eps_loc: np.ndarray
    r_s: np.ndarray
    ghost: np.ndarray
    status: np.ndarray
    beta: np.ndarray
    r: np.ndarray
    row: np.ndarray
    eps: np.ndarray
    i_s: np.ndarray
    grid: tuple


def orbital_count(Z: int, method: int = 0, config=None, charge: float = 0.0) -> int:
    """Orbital rows of one atom in the radial export: its levels (dftatom_aufbau), or alpha plus beta levels (dftatom_split_spin) for
    LSDA (method 1 / 3); for a configured atom (`config` or `charge`, as in Options) its configuration's entries."""
    if config is not None or float(charge) != 0.0:
        return len(Options(int(Z), method=int(method), charge=charge, config=config).entries())
    if int(method) & 1:
        a, b, _, _ = split_spin(Z)
        return len(a) + len(b)
    return len(aufbau(Z))


def _entry4(e, method):
    """(n, l, occ) -> (n, l, 0, occ); (n, l, spin, occ) as given."""
    if len(e) == 3:
        if int(method) & 1:
            raise DFTAtomError(f"configuration entry {tuple(e)}: LSDA entries are (n, l, spin, occ)")
        return (int(e[0]), int(e[1]), 0, float(e[2]))
    if len(e) == 4:
        return (int(e[0]), int(e[1]), int(e[2]), float(e[3]))
    raise DFTAtomError(f"configuration entry {tuple(e)}: expected (n, l, occ) or (n, l, spin, occ)")


def _as_method_form(entries, method):
    return [(n, l, occ) for n, l, _, occ in entries] if not int(method) & 1 else list(entries)


def config_aufbau(Z: int, method: int = 0, charge: float = 0.0):
    """The reference's configuration of atom Z ionised by `charge` electrons (fractional allowed, < 0 = anion; dftatom_config_aufbau):
    (n, l, occ) entries for LDA, (n, l, spin, occ) for LSDA (alpha then beta, each in (n, l) order)."""
    cfg = _CConfig()
    _check(load_library().dftatom_config_aufbau(int(Z), int(method), float(charge), C.byref(cfg)))
    return _as_method_form([(cfg.orb[k].n, cfg.orb[k].l, cfg.orb[k].spin, cfg.orb[k].occ) for k in range(cfg.n_orbitals)], method)


_CORES = {"He": 2, "Ne": 10, "Ar": 18, "Kr": 36, "Xe": 54, "Rn": 86}
_TOKEN = re.compile(r"^(\d)([spdf])((?:\d+(?:\.\d*)?|\.\d+)(?:[eE][-+]?\d+)?)(?:/((?:\d+(?:\.\d*)?|\.\d+)(?:[eE][-+]?\d+)?))?$")


def parse_config(s: str, method: int = 0):
    """A configuration string: whitespace-separated subshells "2p4.5" (n, letter, occupation), in LSDA also "2p3/1" (alpha / beta), and
    the cores [He] [Ne] [Ar] [Kr] [Xe] [Rn] (that atom's reference Aufbau configuration).  A total in LSDA is split like split_spin
    (alpha min(occ, 2l + 1), beta the rest, beta listed only when nonzero).  A subshell given again replaces the earlier one (all of
    its spins): "[Ne] 2p5 3s1" is the excited neon.  Returns the entries in the form Options.config takes for `method`."""
    lsda = bool(int(method) & 1)
    out = []
    for tok in s.split():
        m = re.fullmatch(r"\[([A-Z][a-z])\]", tok)
        if m:
            if m.group(1) not in _CORES:
                raise DFTAtomError(f"configuration {s!r}: unknown core {tok} (use one of {' '.join('[' + k + ']' for k in _CORES)})")
            core = [_entry4(e, method) for e in config_aufbau(_CORES[m.group(1)], method, 0.0)]
            out = [e for e in out if (e[0], e[1]) not in {(c[0], c[1]) for c in core}] + core
            continue
        m = _TOKEN.match(tok)
        if not m:
            raise DFTAtomError(f"configuration {s!r}: cannot read {tok!r} (expected e.g. 3d10, 2p4.5, [Ar]" + (", 2p3/1)" if lsda else ")"))
        n, l = int(m.group(1)), "spdf".index(m.group(2))
        a = float(m.group(3))
        out = [e for e in out if (e[0], e[1]) != (n, l)]
        if m.group(4) is not None:
            if not lsda:
                raise DFTAtomError(f"configuration {s!r}: the alpha/beta form {tok!r} needs LSDA (method 1 or 3)")
            out += [(n, l, 0, a), (n, l, 1, float(m.group(4)))]
        elif lsda:
            up = min(a, float(2 * l + 1))
            out.append((n, l, 0, up))
            if a - up > 0:
                out.append((n, l, 1, a - up))
        else:
            out.append((n, l, 0, a))
    out.sort(key=lambda e: (e[2], e[0], e[1]))
    return _as_method_form(out, method)


def format_config(config, method: int = 0) -> str:
    """The string form of a configuration (inverse of parse_config: parse_config(format_config(c, m), m) == c for entries in the order
    parse_config returns)."""
    e4 = [_entry4(e, method) for e in config]
    beta = {(n, l): occ for n, l, spin, occ in e4 if spin == 1}
    g = lambda x: f"{x:.17g}"
    out = []
    for n, l, spin, occ in e4:
        if spin == 1:
            continue
        sub = f"{n}{'spdf'[l]}"
        out.append(f"{sub}{g(occ)}/{g(beta[(n, l)])}" if (n, l) in beta else f"{sub}{g(occ)}")
    return " ".join(out)


def _levels_from_c(arr, n):
    return [Level(arr[k].n, arr[k].l, arr[k].occ, arr[k].nodes, arr[k].E) for k in range(n)]


def aufbau(Z: int) -> List[Level]:
    """AufbauPrinciple::GetSubshells(Z) sorted by (n,l) (AufbauPrinciple.h:36-75, DFTAtom.cpp:367)."""
    lib = load_library()
    buf = (_CLevel * MAX_LEVELS)()
    n = _check(lib.dftatom_aufbau(int(Z), buf, MAX_LEVELS))
    return _levels_from_c(buf, n)


def split_spin(Z: int):
    """DFTAtom::InitializeLevels (DFTAtom.cpp:611-638): (alpha levels, beta levels, n_alpha, n_beta)."""
    lib = load_library()
    a = (_CLevel * MAX_LEVELS)()
    b = (_CLevel * MAX_LEVELS)()
    na, nb, ea, eb = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    _check(lib.dftatom_split_spin(int(Z), a, C.byref(na), b, C.byref(nb), C.byref(ea), C.byref(eb)))
    return _levels_from_c(a, na.value), _levels_from_c(b, nb.value), ea.value, eb.value


def estimate_cost(Z: int, method: int = 0) -> float:
    """Relative cost of one atom for sharding: (spin) orbitals x expected SCF steps (dftatom_estimate_cost)."""
    return float(load_library().dftatom_estimate_cost(int(Z), int(method)))


def partition(Zs, methods, n_ranks: int):
    """rank of every atom, longest-processing-time-first on dftatom_estimate_cost (dftatom_partition)."""
    z = _i32(Zs); m = _i32(methods); out = np.zeros(len(z), np.int32)
    _check(load_library().dftatom_partition(_i(z), _i(m), len(z), int(n_ranks), _i(out)))
    return [int(x) for x in out]


def n_nodes(levels: int) -> int:
    return load_library().dftatom_n_nodes(int(levels))


def _radial_buffers(n, N, rows):
    """One allocation for the radial export of n atoms with `rows` orbital rows: (the views of _decode, the _CRadial over them)."""
    buf = np.zeros(N + n * 5 * N + n * 2 + rows * (N + N_MOMENTS))      # r | rho | V | V_H | atom moments | orbitals | moments
    r = buf[:N]
    rho = buf[N:N + 2 * n * N].reshape(n, 2, N)
    V = buf[N + 2 * n * N:N + 4 * n * N].reshape(n, 2, N)
    VH = buf[N + 4 * n * N:N + 5 * n * N].reshape(n, N)
    am = buf[N + 5 * n * N:N + 5 * n * N + 2 * n].reshape(n, 2)
    q = N + 5 * n * N + 2 * n
    orb = buf[q:q + rows * N].reshape(rows, N)
    mom = buf[q + rows * N:].reshape(rows, N_MOMENTS)
    return (r, rho, V, VH, am, orb, mom), _CRadial(_d(r), _d(rho), _d(V), _d(VH), _d(orb), rows, _d(mom), _d(am))


def _decode(options, entries, cres, csteps, stride, radial):
    """Result objects of n = len(options) C records (csteps: None or [n][stride] step records; radial: None or the arrays of the
    export (r, rho, V, V_H, atom moments, orbitals, moments)); entries[a]: the (n, l, spin, occ) configuration of atom a or None."""
    n = len(options)
    keep_steps = csteps is not None
    # host structs -> Python objects in bulk (numpy structured views of the ctypes arrays: one pass in C instead of a ctypes
    # attribute access per field)
    ra = np.frombuffer(cres, dtype=_RESULT_DTYPE, count=n)
    head = ra[["status", "n_steps", "n_spin", "Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"]].tolist()
    nlv = ra["n_levels"]
    used = (_LEVEL_IDX < nlv[:, :, None]) & (_SPIN_IDX < ra["n_spin"][:, None, None])        # [atom][spin][k]
    lev, sor = ra["levels"][used].tolist(), ra["sorted"][used].tolist()                        # flat, (n, l, occ, nodes, E) each
    n_levels = nlv.tolist()
    sa = np.frombuffer(csteps, dtype=_STEP_DTYPE, count=n * stride) if keep_steps else None
    out = []
    p = 0
    for a in range(n):
        status, n_steps, n_spin, etot, ekin, ecoul, eenuc, exc = head[a]
        nl = n_levels[a]
        lv, sl = [], []
        for s in range(n_spin):
            q = p + nl[s]
            lv.append(lev[p:q]); sl.append(sor[p:q])
            p = q
        if entries[a] is not None:         # the exact occupations (the C records hold them rounded)
            occ = {(x[0], x[1], x[2]): x[3] for x in entries[a]}
            lv = [[(t[0], t[1], occ[(t[0], t[1], s)]) + tuple(t[3:]) for t in ch] for s, ch in enumerate(lv)]
            sl = [[(t[0], t[1], occ[(t[0], t[1], s)]) + tuple(t[3:]) for t in ch] for s, ch in enumerate(sl)]
        steps = []
        if keep_steps and n_steps:
            blk = sa[a * stride:a * stride + n_steps]
            E = blk["E"].tolist()
            rest = blk[["Etotal", "Ekin", "Ecoul", "Eenuc", "Exc", "levels_converged", "stop_criterion_met"]].tolist()
            for k in range(n_steps):
                r_ = rest[k]
                steps.append(Step([E[k][s][:nl[s]] for s in range(n_spin)], r_[0], r_[1], r_[2], r_[3], r_[4], bool(r_[5]), bool(r_[6])))
        out.append(Result(options[a], status, n_steps, lv, sl, etot, ekin, ecoul, eenuc, exc, steps))
    if radial is not None:
        r, rho, V, VH, am, orb, mom = radial
        row = 0
        for a, res in enumerate(out):
            ns = 2 if options[a].method & 1 else 1
            orbs, moms = [], []
            for s in range(ns):
                k = n_levels[a][s]
                orbs.append(orb[row:row + k]); moms.append(mom[row:row + k])
                row += k
            res.radial = Radial(r, rho[a, :ns], V[a, :ns], VH[a], orbs, moms, float(am[a, 0]), float(am[a, 1]))
    return out


class Context:
    """Owns the CUDA device state behind an opaque dftatom_ctx* (one per GPU / host thread)."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        _check(self._lib.dftatom_create(C.byref(self._h), int(device)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.dftatom_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_option(self, key: str, value: float):
        _check(self._lib.dftatom_set_option(self._h, key.encode(), float(value)))

    # ---- L2 ----
    def solve_batch(self, options: Sequence[Options], keep_steps: bool = True, radial: bool = False) -> List[Result]:
        """One batch of independent atoms (dftatom_solve_batch).  radial=True: every Result also gets `radial` (a Radial: converged
        density, potentials, orbitals and their moments, dftatom_solve_batch_radial).  Atoms with a `charge` or a `config` are solved
        with that configuration (dftatom_solve_batch_config); their Level.occ is the exact occupation."""
        n = len(options)
        copts = (_COptions * n)(*[o._c() for o in options])
        entries = [o.entries() for o in options]
        ccfg = None
        if any(e is not None for e in entries):
            ccfg = (_CConfig * n)()
            for a, e in enumerate(entries):
                if e is None:
                    continue
                if len(e) > 2 * MAX_LEVELS:
                    raise DFTAtomError(f"atom {a} (Z = {options[a].Z}): {len(e)} configuration entries, at most {2 * MAX_LEVELS}")
                ccfg[a].n_orbitals = len(e)
                for k, x in enumerate(e):
                    ccfg[a].orb[k] = _COccupation(*x)
        cres = (_CResult * n)()
        stride = MAX_STEPS_LSDA if any(o.method for o in options) else MAX_STEPS_LDA
        csteps = (_CStep * (n * stride))() if keep_steps else None
        views = None
        if radial and n:
            N = n_nodes(options[0].MultigridLevels)
            rows = sum(len(e) if e is not None else orbital_count(o.Z, o.method) for o, e in zip(options, entries))
            views, crad = _radial_buffers(n, N, rows)
            _check(self._lib.dftatom_solve_batch_config(self._h, copts, ccfg, n, cres, csteps, stride if keep_steps else 0, C.byref(crad)))
        elif ccfg is not None:
            _check(self._lib.dftatom_solve_batch_config(self._h, copts, ccfg, n, cres, csteps, stride if keep_steps else 0, None))
        else:
            _check(self._lib.dftatom_solve_batch(self._h, copts, n, cres, csteps, stride if keep_steps else 0))
        return _decode(options, entries, cres, csteps if keep_steps else None, stride, views)

    def solve_pseudo_batch(self, pseudos, configs, mixing: float = 0.5, method: int = 0, keep_steps: bool = True,
                           radial: bool = False) -> List[Result]:
        """Self-consistent pseudo-atoms (dftatom_solve_pseudo_batch).  pseudos: Pseudopotential objects (Context.tm_pseudize /
        Context.pseudize, with `n` set), one pseudo-atom each: its channels (one per l) with ionic potentials V_ion, reference principal
        numbers n and ionic charge z_val = sum of the channels' occupations.  configs: valence configurations with all-electron labels,
        parse_config strings or entry lists ((n, l, occ) for LDA, (n, l, spin, occ) for LSDA), broadcast against pseudos.  All pseudos
        share one grid (the logarithmic grid).  Returns one Result per pseudo-atom: levels with the all-electron n and nodes = n - n_ref,
        Eenuc = E_ion, Ecoul = E_H, Exc, Ekin and Etotal as documented there; options = Options(Z = round(z_val), the grid, mixing,
        method, config = the entries).  radial=True: Result.radial with V = the screening V_H + V_xc per spin.  A pseudopotential with
        rho_pc (unscreened with a partial core) is solved with that core (dftatom_solve_pseudo_batch_core); batches may mix both kinds."""
        pseudos = list(pseudos) if isinstance(pseudos, (list, tuple)) else [pseudos]
        one = isinstance(configs, str) or (len(configs) > 0 and all(isinstance(e, (list, tuple)) and len(e) in (3, 4)
                                                                     and not isinstance(e[0], (list, tuple, str)) for e in configs))
        configs = [configs] if one else list(configs)
        n = max(len(pseudos), len(configs))
        if len(pseudos) not in (1, n) or len(configs) not in (1, n):
            raise DFTAtomError(f"solve_pseudo_batch: {len(pseudos)} pseudopotentials and {len(configs)} configurations do not broadcast")
        pseudos = pseudos * (n // len(pseudos)); configs = configs * (n // len(configs))
        grid = pseudos[0].grid
        if grid is None or any(pp.grid != grid for pp in pseudos):
            raise DFTAtomError("solve_pseudo_batch: every Pseudopotential must come from Context.tm_pseudize on one grid")
        levels, delta, max_r = grid
        rows, row_of, catoms = [], {}, (_CPseudoAtom * n)()
        pc_rows, pc_of, pc_row = [], {}, np.full(n, -1, dtype=np.int32)
        for a, pp in enumerate(pseudos):
            if pp.n is None:
                raise DFTAtomError(f"solve_pseudo_batch: pseudopotential {a} has no reference principal numbers (Pseudopotential.n)")
            if len(set(pp.l.tolist())) != len(pp.l):
                raise DFTAtomError(f"solve_pseudo_batch: pseudopotential {a} has two channels of one l")
            key = id(pp)
            if key not in row_of:
                row_of[key] = len(rows)
                rows += [pp.V_ion[c] for c in range(len(pp.l))]
            base = row_of[key]
            catoms[a].row[:] = [-1] * 4
            catoms[a].n_ref[:] = [0] * 4
            for c, l in enumerate(pp.l.tolist()):
                catoms[a].row[l] = base + c
                catoms[a].n_ref[l] = int(pp.n[c])
            if pp.rho_pc is not None:
                pots = set(np.asarray(pp.pot).tolist())
                if len(pots) != 1:
                    raise DFTAtomError(f"solve_pseudo_batch: pseudopotential {a} with a core has channels on several potential rows")
                if key not in pc_of:
                    pc_of[key] = len(pc_rows)
                    pc_rows.append(np.asarray(pp.rho_pc)[pots.pop()])
                pc_row[a] = pc_of[key]
            catoms[a].z_val = float(np.sum(pp.occ))
            catoms[a].mixing = float(mixing)
            catoms[a].method = int(method)
        entries = [[_entry4(e, method) for e in (parse_config(c, method) if isinstance(c, str) else c)] for c in configs]
        ccfg = (_CConfig * n)()
        for a, e in enumerate(entries):
            if len(e) > 2 * MAX_LEVELS:
                raise DFTAtomError(f"atom {a}: {len(e)} configuration entries, at most {2 * MAX_LEVELS}")
            ccfg[a].n_orbitals = len(e)
            for k, x in enumerate(e):
                ccfg[a].orb[k] = _COccupation(*x)
        V = _f64(np.array(rows))
        cres = (_CResult * n)()
        stride = MAX_STEPS_LSDA if method & 1 else MAX_STEPS_LDA
        csteps = (_CStep * (n * stride))() if keep_steps else None
        views, crad = _radial_buffers(n, V.shape[1], sum(len(e) for e in entries)) if radial else (None, None)
        if pc_rows:
            PC = _f64(np.array(pc_rows))
            _check(self._lib.dftatom_solve_pseudo_batch_core(self._h, int(levels), float(delta), float(max_r), _d(V), V.shape[0], catoms, ccfg, n,
                                                             cres, csteps, stride if keep_steps else 0, C.byref(crad) if radial else None,
                                                             _d(PC), PC.shape[0], _i(pc_row)))
        else:
            _check(self._lib.dftatom_solve_pseudo_batch(self._h, int(levels), float(delta), float(max_r), _d(V), V.shape[0], catoms, ccfg, n,
                                                        cres, csteps, stride if keep_steps else 0, C.byref(crad) if radial else None))
        options = [Options(int(round(catoms[a].z_val)), int(levels), float(max_r), float(delta), float(mixing), int(method),
                           config=_as_method_form(entries[a], method)) for a in range(n)]
        return _decode(options, entries, cres, csteps, stride, views)


    def last_timing(self):
        ms, n = C.c_double(), C.c_longlong()
        _check(self._lib.dftatom_last_timing(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def last_graph_iterations(self) -> int:
        """SCF steps the last solve_batch ran inside the CUDA-graph while node (0: host-driven loop)."""
        v = C.c_longlong()
        _check(self._lib.dftatom_last_graph_iterations(self._h, C.byref(v)))
        return v.value

    def last_transfer(self):
        """(host->device bytes, device->host bytes) of the last solve_batch."""
        a, b = C.c_longlong(), C.c_longlong()
        _check(self._lib.dftatom_last_transfer(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def last_profile(self):
        """Per-kernel-class {ms, launches, work} of the last solve_batch (needs set_option('profile', 1))."""
        buf = (_CProfile * len(KERNEL_CLASSES))()
        _check(self._lib.dftatom_last_profile(self._h, buf))
        return {k: dict(ms=buf[i].ms, launches=buf[i].launches, work=buf[i].work) for i, k in enumerate(KERNEL_CLASSES)}

    def measure_fp64_peak(self) -> float:
        v = C.c_double()
        _check(self._lib.dftatom_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    # ---- L1 components ----
    def numerov_lanes(self, V, levels, delta, max_r, l, E, nodes_limit, impl=1):
        """impl=1: reference-shaped sweep (count = CountNodes); impl=0: production sweep (count = full Sturm count)."""
        V = _f64(V); l = _i32(l); E = _f64(E); lim = _i32(nodes_limit)
        n = len(E)
        sign = np.zeros(n, np.int32); lg = np.zeros(n, np.float64); cnt = np.zeros(n, np.int32)
        _check(self._lib.dftatom_numerov_lanes(self._h, _d(V), int(levels), float(delta), float(max_r), n, _i(l), _d(E), _i(lim), int(impl),
                                               _i(sign), _d(lg), _i(cnt)))
        return sign, lg, cnt

    def numerov_lanes_timed(self, V, levels, delta, max_r, l, E, nodes_limit, impl=0, reps=10):
        """numerov_lanes plus (ms per launch over `reps` device-timed launches, lane node-steps per launch)."""
        V = _f64(V); l = _i32(l); E = _f64(E); lim = _i32(nodes_limit)
        n = len(E)
        sign = np.zeros(n, np.int32); lg = np.zeros(n, np.float64); cnt = np.zeros(n, np.int32)
        ms = C.c_float(); ns = C.c_double()
        _check(self._lib.dftatom_numerov_lanes_timed(self._h, _d(V), int(levels), float(delta), float(max_r), n, _i(l), _d(E), _i(lim), int(impl),
                                                     _i(sign), _d(lg), _i(cnt), int(reps), C.byref(ms), C.byref(ns)))
        return sign, lg, cnt, ms.value, ns.value

    def level_search(self, V, levels, delta, max_r, Z, n, l):
        V = _f64(V); n = _i32(n); l = _i32(l)
        E = np.zeros(len(n), np.float64); ok = np.zeros(len(n), np.int32)
        _check(self._lib.dftatom_level_search(self._h, _d(V), int(levels), float(delta), float(max_r), int(Z), len(n), _i(n), _i(l), _d(E), _i(ok)))
        return E, ok

    def numerov_orbital(self, V, levels, delta, max_r, l, E):
        V = _f64(V)
        u = np.zeros(len(V), np.float64); mp = C.c_int()
        _check(self._lib.dftatom_numerov_orbital(self._h, _d(V), int(levels), float(delta), float(max_r), int(l), float(E), _d(u), C.byref(mp)))
        return u, mp.value

    def poisson_solve(self, levels, delta, max_r, Z, rho):
        rho = _f64(np.atleast_2d(rho)); Z = _i32(np.atleast_1d(Z))
        U = np.zeros_like(rho); used = np.zeros(len(Z), np.int32)
        _check(self._lib.dftatom_poisson_solve(self._h, int(levels), float(delta), float(max_r), len(Z), _i(Z), _d(rho), _d(U), _i(used)))
        return U, used

    def poisson_increment(self, levels, delta, max_r, rho, rho_prev, U, skip=None, solver=0, n_vcycles=7):
        """One warm Poisson solve of the SCF in increment form (dftatom_poisson_increment): solver 0 direct, 1 warm V-cycles,
        2 V-cycles of the cold solvers.  Returns (U + dU, rho_prev after the call = rho except where skipped); the inputs are not changed."""
        rho = _f64(np.atleast_2d(rho)); rho_prev = _f64(np.atleast_2d(rho_prev)).copy(); U = _f64(np.atleast_2d(U)).copy()
        if rho.shape != rho_prev.shape or rho.shape != U.shape or rho.shape[1] != (1 << int(levels)) + 1:
            raise ValueError("rho, rho_prev and U must have the same shape [n_dens][2^levels + 1]")
        sk = None if skip is None else _i32(np.asarray(skip).astype(np.int32))
        if sk is not None and len(sk) != rho.shape[0]:
            raise ValueError("skip must have one entry per density")
        _check(self._lib.dftatom_poisson_increment(self._h, int(levels), float(delta), float(max_r), rho.shape[0], _d(rho), _d(rho_prev), _d(U),
                                                   None if sk is None else _i(sk), int(solver), int(n_vcycles)))
        return U, rho_prev

    def poisson_vcycles(self, levels, delta, phi, src, n_cycles):
        phi = _f64(np.atleast_2d(phi)).copy(); src = _f64(np.atleast_2d(src))
        err = np.zeros(phi.shape[0], np.float64)
        _check(self._lib.dftatom_poisson_vcycles(self._h, int(levels), float(delta), phi.shape[0], _d(phi), _d(src), int(n_cycles), _d(err)))
        return phi, err

    def poisson_scratch_bytes(self, levels, n_dens) -> int:
        return int(self._lib.dftatom_poisson_scratch_bytes(int(levels), int(n_dens)))

    def poisson_vcycles_dev(self, levels, delta, n_dens, d_phi, d_src, ld, d_scratch, scratch_bytes, n_cycles, fuse_tops=True):
        """Stream-mode V-cycles on DEVICE arrays (addresses as ints, e.g. torch.Tensor.data_ptr()): phi[n_dens][ld] in place,
        src[n_dens][ld]; returns (device ms, kernel launches).  levels >= 15 (config C5a)."""
        ms, nl = C.c_float(), C.c_longlong()
        _check(self._lib.dftatom_poisson_vcycles_dev(self._h, int(levels), float(delta), int(n_dens), C.c_void_p(int(d_phi)), C.c_void_p(int(d_src)),
                                                     int(ld), C.c_void_p(int(d_scratch)), int(scratch_bytes), int(n_cycles), int(bool(fuse_tops)),
                                                     C.byref(ms), C.byref(nl)))
        return ms.value, nl.value

    def vwn(self, rho_a, rho_b=None):
        ra = _f64(rho_a); n = len(ra)
        vexc = np.zeros(n); edif = np.zeros(n)
        if rho_b is None:
            _check(self._lib.dftatom_vwn(self._h, n, _d(ra), None, None, None, _d(vexc), _d(edif)))
            return vexc, edif
        rb = _f64(rho_b); va = np.zeros(n); vb = np.zeros(n)
        _check(self._lib.dftatom_vwn(self._h, n, _d(ra), _d(rb), _d(va), _d(vb), _d(vexc), _d(edif)))
        return va, vb, vexc, edif

    def xc_lda(self, functional, rho):
        """(Vexc, eps_xc - Vexc) by functional: 0 VWN, 1 Chachiyo, 2 Chachiyo improved (ExcCor.h:27-95)."""
        r = _f64(rho); n = len(r)
        vexc = np.zeros(n); edif = np.zeros(n)
        _check(self._lib.dftatom_xc_lda(self._h, int(functional), n, _d(r), _d(vexc), _d(edif)))
        return vexc, edif

    def radial_moments(self, levels, delta, max_r, u):
        """[n_rows][N_MOMENTS] moments <1/r>, <r>, <r^2> of the rows of u (used as given) on the grid (levels, delta, max_r; delta 0:
        uniform), with the quadrature of the radial export (dftatom_radial_moments)."""
        u = _f64(np.atleast_2d(u))
        out = np.zeros((u.shape[0], N_MOMENTS))
        _check(self._lib.dftatom_radial_moments(self._h, int(levels), float(delta), float(max_r), _d(u), u.shape[0], _d(out)))
        return out

    def log_derivatives(self, V, levels, delta, max_r, pot, l, r_c, E) -> LogDerivatives:
        """D_l(E) = u'(r_c) / u(r_c) of the outward radial solution for every (channel, energy) (dftatom_log_derivatives).  V: [n_pot][N]
        potentials (one row may be given as [N]), e.g. rows of Result.radial.V; channel c = (V row pot[c], l[c], r_c[c] in bohr): pot, l
        and r_c are broadcast against each other; E: energies shared by all channels."""
        V = _f64(np.atleast_2d(V))
        pot, l, r_c = np.broadcast_arrays(np.atleast_1d(pot), np.atleast_1d(l), np.atleast_1d(r_c))
        pot = _i32(pot); l = _i32(l); r_c = _f64(r_c); E = _f64(np.atleast_1d(E))
        nc, ne = len(pot), len(E)
        out = np.zeros(nc * ne, dtype=np.dtype(_CLogDeriv))
        used = np.zeros(nc)
        _check(self._lib.dftatom_log_derivatives(self._h, int(levels), float(delta), float(max_r), _d(V), V.shape[0], _i(pot), _i(l), _d(r_c), nc,
                                                 _d(E), ne, out.ctypes.data_as(C.POINTER(_CLogDeriv)), _d(used)))
        out = out.reshape(nc, ne)
        return LogDerivatives(out["D"].copy(), out["u"].copy(), out["du"].copy(), out["nodes"].copy(), used, E.copy())

    def tm_pseudize(self, V, u, levels, delta, max_r, pot, orbital, l, eps, occ, r_c, n=None, rho_pc=None) -> Pseudopotential:
        """Troullier-Martins pseudization and unscreening (dftatom_tm_pseudize).  V: [n_pot][N] potentials, u: [n_orb][N] all-electron
        orbitals (one row of either may be given as [N]), e.g. rows of Result.radial.V and Result.radial.orbitals; channel c = (V row pot[c],
        u row orbital[c], l[c], eigenvalue eps[c], occupation occ[c], radius r_c[c] in bohr), broadcast against each other.  The channels
        sharing a potential row are one pseudo-atom for the unscreening.  n (optional, broadcast likewise): the all-electron principal
        number of every channel's reference state, kept as Pseudopotential.n.  rho_pc (optional, [n_pot][N]): a partial core density per
        potential row; the unscreening then removes V_xc(rho_val + rho_pc) (dftatom_tm_pseudize_core), kept as Pseudopotential.rho_pc."""
        V = _f64(np.atleast_2d(V)); u = _f64(np.atleast_2d(u))
        pc = None if rho_pc is None else _f64(np.atleast_2d(rho_pc))
        if pc is not None and pc.shape != V.shape:
            raise ValueError(f"tm_pseudize: rho_pc has shape {pc.shape}, V {V.shape}")
        pot, orbital, l, eps, occ, r_c = np.broadcast_arrays(*(np.atleast_1d(x) for x in (pot, orbital, l, eps, occ, r_c)))
        nc, N = len(pot), V.shape[1]
        ch = np.zeros(nc, dtype=np.dtype(_CTmChannel))
        ch["pot"], ch["orbital"], ch["l"], ch["eps"], ch["occ"], ch["r_c"] = pot, orbital, l, eps, occ, r_c
        res = np.zeros(nc, dtype=np.dtype(_CTmResult))
        u_ps, v_scr, v_ion = (np.zeros((nc, N)) for _ in range(3))
        rho = np.zeros((V.shape[0], N))
        _check(self._lib.dftatom_tm_pseudize_core(self._h, int(levels), float(delta), float(max_r), _d(V), V.shape[0], _d(u), u.shape[0],
                                                  ch.ctypes.data_as(C.POINTER(_CTmChannel)), nc, res.ctypes.data_as(C.POINTER(_CTmResult)),
                                                  _d(u_ps), _d(v_scr), _d(v_ion), _d(rho), None if pc is None else _d(pc)))
        rr = np.zeros(N)                                    # the engine's node radii
        _check(self._lib.dftatom_grid_nodes(self._h, int(levels), float(delta), float(max_r), _d(rr)))
        nn = None if n is None else _i32(np.broadcast_to(np.atleast_1d(n), (nc,))).copy()
        return Pseudopotential(_i32(l).copy(), _f64(eps).copy(), _f64(occ).copy(), res["r_c"].copy(), res["c"].copy(), res["q"].copy(),
                               res["status"].copy(), rr, u_ps, v_scr, v_ion, rho, _i32(pot).copy(), (int(levels), float(delta), float(max_r)), nn,
                               None, None if pc is None else pc.copy())

    def partial_core(self, u, levels, delta, max_r, row, orbital, occ, r_pc) -> PartialCore:
        """Core densities and Louie-Froyen-Cohen partial cores (dftatom_partial_core).  u: [n_orb][N] all-electron orbitals; core entry k =
        (output row row[k], u row orbital[k], occupation occ[k]), broadcast against each other; r_pc: [n_rows] radii (0 = the full core),
        one per output row."""
        u = _f64(np.atleast_2d(u))
        r_pc = _f64(np.atleast_1d(r_pc))
        row, orbital, occ = np.broadcast_arrays(*(np.atleast_1d(x) for x in (row, orbital, occ)))
        nr, N = len(r_pc), u.shape[1]
        ce = np.zeros(len(row), dtype=np.dtype(_CCoreOrbital))
        ce["row"], ce["orbital"], ce["occ"] = row, orbital, occ
        res = np.zeros(nr, dtype=np.dtype(_CPccResult))
        rho_core, rho_pc = np.zeros((nr, N)), np.zeros((nr, N))
        _check(self._lib.dftatom_partial_core(self._h, int(levels), float(delta), float(max_r), _d(u), u.shape[0],
                                              ce.ctypes.data_as(C.POINTER(_CCoreOrbital)), len(ce), _d(r_pc), nr,
                                              res.ctypes.data_as(C.POINTER(_CPccResult)), _d(rho_core), _d(rho_pc)))
        rr = np.zeros(N)
        _check(self._lib.dftatom_grid_nodes(self._h, int(levels), float(delta), float(max_r), _d(rr)))
        return PartialCore(res["r_pc"].copy(), res["i_pc"].copy(), res["A"].copy(), res["B"].copy(), res["n_core"].copy(), res["n_pc"].copy(),
                           res["status"].copy(), rho_core, rho_pc, rr)

    def pseudize(self, result, r_c, r_pc=None) -> Pseudopotential:
        """Pseudopotentials of a solved LDA atom (Result of solve_batch(..., radial=True)): for every l of result.levels[0] the level of
        largest n is the valence channel, with its eigenvalue and occupation.  r_c: one radius, a sequence indexed by l, or a dict {l: r_c}.
        r_pc (optional; 0 = the full core): unscreen with the nonlinear core correction, the partial core of the other (core) levels at
        r_pc (Context.partial_core); the result carries rho_core, rho_pc and core.  DFTAtomError when the core density does not decrease at
        r_pc (no partial core there)."""
        o = result.options
        if result.radial is None:
            raise ValueError("pseudize needs the radial state: solve with radial=True")
        if o.method & 1:
            raise ValueError("pseudize needs an LDA atom (method 0 or 2): the unscreening is spin-unpolarised")
        best = {}
        for k, lev in enumerate(result.levels[0]):
            if lev.l not in best or lev.n > result.levels[0][best[lev.l]].n:
                best[lev.l] = k
        ls = sorted(best)
        if isinstance(r_c, dict):
            rcs = [r_c[l] for l in ls]
        elif np.ndim(r_c) == 0:
            rcs = [float(r_c)] * len(ls)
        else:
            rcs = [r_c[l] for l in ls]
        lev = [result.levels[0][best[l]] for l in ls]
        rad = result.radial
        grid = (o.MultigridLevels, 0.0 if o.method >= 2 else o.deltaGrid, o.MaxR)
        pc = None
        if r_pc is not None:
            core = [k for k, x in enumerate(result.levels[0]) if k not in best.values()]
            pc = self.partial_core(rad.orbitals[0], *grid, 0, core, [float(result.levels[0][k].occ) for k in core], [float(r_pc)])
            if pc.status[0] != 0:
                raise DFTAtomError(f"pseudize: the core density does not decrease at r_pc = {pc.r_pc[0]!r}: no partial core there")
        pp = self.tm_pseudize(rad.V[0], rad.orbitals[0], *grid, 0, [best[l] for l in ls], ls, [x.E for x in lev], [float(x.occ) for x in lev],
                              rcs, [x.n for x in lev], rho_pc=None if pc is None else pc.rho_pc)
        if pc is not None:
            pp.rho_core, pp.core = pc.rho_core, pc
        return pp

    def kb_form(self, V, u, levels, delta, max_r, row, loc, l, eps) -> KleinmanBylander:
        """Kleinman-Bylander form and GSS ghost test (dftatom_kb_form).  V: [n_rows][N] screened potentials, u: [n_rows][N] pseudo-orbitals
        (e.g. Pseudopotential.V_scr and .u); channel c = (row[c], local row loc[c], l[c], reference eigenvalue eps[c]), broadcast against
        each other."""
        V = _f64(np.atleast_2d(V)); u = _f64(np.atleast_2d(u))
        row, loc, l, eps = np.broadcast_arrays(*(np.atleast_1d(x) for x in (row, loc, l, eps)))
        nc, N = len(row), V.shape[1]
        ch = np.zeros(nc, dtype=np.dtype(_CKbChannel))
        ch["row"], ch["loc"], ch["l"], ch["eps"] = row, loc, l, eps
        res = np.zeros(nc, dtype=np.dtype(_CKbResult))
        beta = np.zeros((nc, N))
        _check(self._lib.dftatom_kb_form(self._h, int(levels), float(delta), float(max_r), _d(V), _d(u), V.shape[0],
                                         ch.ctypes.data_as(C.POINTER(_CKbChannel)), nc, res.ctypes.data_as(C.POINTER(_CKbResult)), _d(beta)))
        rr = np.zeros(N)
        _check(self._lib.dftatom_grid_nodes(self._h, int(levels), float(delta), float(max_r), _d(rr)))
        return KleinmanBylander(_i32(l).copy(), _i32(loc).copy(), res["E_KB"].copy(), res["cos"].copy(), res["eps_loc"].copy(), res["r_s"].copy(),
                                res["ghost"].copy(), res["status"].copy(), beta, rr, _i32(row).copy(), _f64(eps).copy(), res["i_s"].copy(),
                                (int(levels), float(delta), float(max_r)))

    def kleinman_bylander(self, pp, l_loc) -> KleinmanBylander:
        """The KB form of a Pseudopotential (Context.tm_pseudize / Context.pseudize): within each potential row the channel of l = l_loc
        is the local potential of the row's other channels."""
        if pp.grid is None:
            raise ValueError("kleinman_bylander needs a Pseudopotential of Context.tm_pseudize")
        loc = np.empty(len(pp.l), np.int32)
        for c, p in enumerate(pp.pot):
            hit = np.nonzero((pp.pot == p) & (pp.l == int(l_loc)))[0]
            if len(hit) == 0:
                raise ValueError(f"l_loc = {l_loc} is not a channel of potential row {p} (channels l = {sorted(pp.l[pp.pot == p].tolist())})")
            loc[c] = hit[0]
        return self.kb_form(pp.V_scr, pp.u, *pp.grid, np.arange(len(pp.l)), loc, pp.l, pp.eps)

    def kb_log_derivatives(self, kb, V_loc, r_c, E) -> LogDerivatives:
        """Logarithmic derivatives of the KB Hamiltonian of every channel of `kb` (dftatom_kb_log_derivatives): local potential row
        kb.loc[c] of V_loc (the V given to kb_form), projector kb.beta[c] with E_KB[c] (none for the local channels), l[c]; r_c broadcast
        over the channels; E shared by all channels."""
        if np.any(kb.status == 2):
            raise ValueError("channels " + str(np.nonzero(kb.status == 2)[0].tolist()) + " have no KB projector (status 2)")
        V = _f64(np.atleast_2d(V_loc)); E = _f64(np.atleast_1d(E))
        nc, ne = len(kb.l), len(E)
        local = kb.status == 1
        ch = np.zeros(nc, dtype=np.dtype(_CKbLdChannel))
        ch["pot"], ch["proj"], ch["l"] = kb.loc, np.where(local, -1, np.arange(nc)), kb.l
        ch["E_KB"], ch["r_c"] = np.where(local, 0.0, kb.E_KB), np.broadcast_to(np.atleast_1d(r_c), (nc,))
        beta = _f64(kb.beta)
        out = np.zeros(nc * ne, dtype=np.dtype(_CLogDeriv))
        used = np.zeros(nc)
        levels, delta, max_r = kb.grid
        _check(self._lib.dftatom_kb_log_derivatives(self._h, int(levels), float(delta), float(max_r), _d(V), V.shape[0], _d(beta), beta.shape[0],
                                                    ch.ctypes.data_as(C.POINTER(_CKbLdChannel)), nc, _d(E), ne,
                                                    out.ctypes.data_as(C.POINTER(_CLogDeriv)), _d(used)))
        out = out.reshape(nc, ne)
        return LogDerivatives(out["D"].copy(), out["u"].copy(), out["du"].copy(), out["nodes"].copy(), used, E.copy())

    def integrate(self, rule, step, v):
        """Integral.h quadratures by rule: 0 Trapezoid, 1 SimpsonOneThird, 2 Simpson38, 3 Boole, 4 Romberg; one result per row of v."""
        v = _f64(np.atleast_2d(v))
        out = np.zeros(v.shape[0])
        _check(self._lib.dftatom_integrate(self._h, int(rule), float(step), _d(v), v.shape[1], v.shape[0], _d(out)))
        return out

    def simpson38(self, step, v):
        v = _f64(np.atleast_2d(v))
        out = np.zeros(v.shape[0])
        _check(self._lib.dftatom_simpson38(self._h, float(step), _d(v), v.shape[1], v.shape[0], _d(out)))
        return out


_default_ctx: Optional[Context] = None


def _ctx() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("DFTATOM_USE_LOCAL_RANK") else 0)
    return _default_ctx


class DFTAtom:
    """Mirror of the reference's `DFT::DFTAtom` static interface (DFTAtom.h:14,17): same names, same argument
    order and meaning; prints the same report to stdout and additionally returns the `Result`."""

    @staticmethod
    def CalculateNonUniformLDA(Z, MultigridLevels, alpha, MaxR, deltaGrid, out=None) -> Result:
        return DFTAtom._run(Options(Z, MultigridLevels, MaxR, deltaGrid, alpha, 0), out)

    @staticmethod
    def CalculateNonUniformLSDA(Z, MultigridLevels, alpha, MaxR, deltaGrid, out=None) -> Result:
        return DFTAtom._run(Options(Z, MultigridLevels, MaxR, deltaGrid, alpha, 1), out)

    @staticmethod
    def CalculateUniformLDA(Z, MultigridLevels, alpha, MaxR, out=None) -> Result:
        """DFTAtom.h:15 (DFTAtom.cpp:60-210): the uniform grid r_i = i MaxR / (N - 1)."""
        return DFTAtom._run(Options(Z, MultigridLevels, MaxR, 0.0, alpha, 2), out)

    @staticmethod
    def CalculateUniformLSDA(Z, MultigridLevels, alpha, MaxR, out=None) -> Result:
        """DFTAtom.h:18 (DFTAtom.cpp:646-844)."""
        return DFTAtom._run(Options(Z, MultigridLevels, MaxR, 0.0, alpha, 3), out)

    @staticmethod
    def _run(opt, out):
        res = _ctx().solve_batch([opt])[0]
        (out or sys.stdout).write(res.report())
        return res
