"""ctypes binding of include/dftatom_b200.h and the Python mirror of the reference's solver surface."""
import ctypes as C
import os
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
    lib.dftatom_radial_moments.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp, C.c_int, _dp]
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

    def _c(self):
        return _COptions(int(self.Z), int(self.MultigridLevels), float(self.MaxR), float(self.deltaGrid), float(self.alpha), int(self.method))


@dataclass
class Level:
    n: int
    l: int
    occ: int
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


def orbital_count(Z: int, method: int = 0) -> int:
    """Orbital rows of one atom in the radial export: its levels (dftatom_aufbau), or alpha plus beta levels (dftatom_split_spin) for
    LSDA (method 1 / 3)."""
    if int(method) & 1:
        a, b, _, _ = split_spin(Z)
        return len(a) + len(b)
    return len(aufbau(Z))


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
        density, potentials, orbitals and their moments, dftatom_solve_batch_radial)."""
        n = len(options)
        copts = (_COptions * n)(*[o._c() for o in options])
        cres = (_CResult * n)()
        stride = MAX_STEPS_LSDA if any(o.method for o in options) else MAX_STEPS_LDA
        csteps = (_CStep * (n * stride))() if keep_steps else None
        if radial and n:
            N = n_nodes(options[0].MultigridLevels)
            rows = sum(orbital_count(o.Z, o.method) for o in options)
            buf = np.zeros(N + n * 5 * N + n * 2 + rows * (N + N_MOMENTS))      # r | rho | V | V_H | atom moments | orbitals | moments
            r = buf[:N]
            rho = buf[N:N + 2 * n * N].reshape(n, 2, N)
            V = buf[N + 2 * n * N:N + 4 * n * N].reshape(n, 2, N)
            VH = buf[N + 4 * n * N:N + 5 * n * N].reshape(n, N)
            am = buf[N + 5 * n * N:N + 5 * n * N + 2 * n].reshape(n, 2)
            q = N + 5 * n * N + 2 * n
            orb = buf[q:q + rows * N].reshape(rows, N)
            mom = buf[q + rows * N:].reshape(rows, N_MOMENTS)
            crad = _CRadial(_d(r), _d(rho), _d(V), _d(VH), _d(orb), rows, _d(mom), _d(am))
            _check(self._lib.dftatom_solve_batch_radial(self._h, copts, n, cres, csteps, stride if keep_steps else 0, C.byref(crad)))
        else:
            _check(self._lib.dftatom_solve_batch(self._h, copts, n, cres, csteps, stride if keep_steps else 0))
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
            steps = []
            if keep_steps and n_steps:
                blk = sa[a * stride:a * stride + n_steps]
                E = blk["E"].tolist()
                rest = blk[["Etotal", "Ekin", "Ecoul", "Eenuc", "Exc", "levels_converged", "stop_criterion_met"]].tolist()
                for k in range(n_steps):
                    r_ = rest[k]
                    steps.append(Step([E[k][s][:nl[s]] for s in range(n_spin)], r_[0], r_[1], r_[2], r_[3], r_[4], bool(r_[5]), bool(r_[6])))
            out.append(Result(options[a], status, n_steps, lv, sl, etot, ekin, ecoul, eenuc, exc, steps))
        if radial and n:
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
