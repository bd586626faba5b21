"""TEST INFRASTRUCTURE: the exact solution of one warm Poisson solve in increment form (dftatom_poisson_increment),

    -a dU_{i-1} + dU_i - b dU_{i+1} = psrc_i (rho_i - rho_prev_i) / 2,   a = (1 + delta/2)/2,   b = (1 - delta/2)/2,   dU_0 = dU_{N-1} = 0,

solved in __float128 by tests/poisson_increment_ref.c, which is compiled on first use into a temporary directory (the tree may be read-only
where tests run).  Two independent solves check it (tests/test_poisson_increment_host.py): exact rationals (small grids) and FP64
scipy.linalg.solve_banded (every grid, to FP64's error)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction

import numpy as np

import oracle_lib as O

_dp = C.POINTER(C.c_double)
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="dftatom_poisson_increment_ref_")
        atexit.register(shutil.rmtree, tmp, True)
        path = os.path.join(tmp, "libpoisson_increment_ref.so")
        cc = shutil.which("cc") or shutil.which("gcc") or "gcc"
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "poisson_increment_ref.c")
        subprocess.run([cc, "-std=gnu11", "-O2", "-fPIC", "-shared", "-o", path, src, "-lm"], check=True)
        L = C.CDLL(path)
        L.inc_psrc.argtypes = [C.c_int, C.c_double, C.c_double, _dp]
        L.inc_solve_h.argtypes = [C.c_int, C.c_double, _dp, _dp]
        L.inc_solve.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, _dp, _dp, _dp]
        _lib = L
    return _lib


def _d(a):
    return a.ctypes.data_as(_dp)


def coefficients(delta):
    """(a, b) as the kernels form them in FP64."""
    return 0.5 * (1.0 + 0.5 * delta), 0.5 * (1.0 - 0.5 * delta)


def psrc(levels, delta, max_r):
    """The grid's source factor r_i 4 pi K_i, built as engine.cpp get_grid builds it (delta = 0: uniform grid)."""
    out = np.zeros((1 << levels) + 1)
    lib().inc_psrc(int(levels), float(delta), float(max_r), _d(out))
    return out


def rhs(levels, delta, max_r, rho, rho_prev):
    """h = psrc (rho - rho_prev) / 2 in FP64 (h_0 = h_{N-1} = 0)."""
    return 0.5 * (psrc(levels, delta, max_r) * (np.asarray(rho, np.float64) - np.asarray(rho_prev, np.float64)))


def solve(levels, delta, max_r, rho, rho_prev):
    """dU [n_dens][N] of densities rho, rho_prev [n_dens][N], h formed and the system solved in __float128, rounded to FP64 once."""
    rho = np.ascontiguousarray(np.atleast_2d(rho), np.float64)
    rho_prev = np.ascontiguousarray(np.atleast_2d(rho_prev), np.float64)
    assert rho.shape == rho_prev.shape and rho.shape[1] == (1 << levels) + 1
    dU = np.zeros_like(rho)
    lib().inc_solve(int(levels), float(delta), float(max_r), rho.shape[0], _d(rho), _d(rho_prev), _d(dU))
    return dU


def solve_h(delta, h):
    """dU of the system with right-hand side h (FP64), solved in __float128."""
    h = np.ascontiguousarray(h, np.float64)
    dU = np.zeros_like(h)
    lib().inc_solve_h(len(h), float(delta), _d(h), _d(dU))
    return dU


def solve_fraction(delta, h):
    """The same system in exact rational arithmetic (Thomas algorithm on Fractions): small grids only."""
    a, b = (Fraction(x) for x in coefficients(delta))
    n = len(h)
    gam = [Fraction(0)] * n
    dl = [Fraction(0)] * n
    for i in range(1, n - 1):
        w = 1 / (1 - a * gam[i - 1])
        gam[i] = b * w
        dl[i] = w * (Fraction(float(h[i])) + a * dl[i - 1])
    x = [Fraction(0)] * n
    for i in range(n - 2, 0, -1):
        x[i] = gam[i] * x[i + 1] + dl[i]
    return x


def solve_banded_fp64(delta, h):
    """The same system by scipy.linalg.solve_banded in FP64 (the form pseudo_ref.hartree_U uses)."""
    from scipy.linalg import solve_banded
    a, b = coefficients(delta)
    m = len(h) - 2
    ab = np.zeros((3, m))
    ab[0, 1:] = -b
    ab[1, :] = 1.0
    ab[2, :-1] = -a
    out = np.zeros(len(h))
    out[1:-1] = solve_banded((1, 1), ab, np.asarray(h[1:-1], np.float64))
    return out


# the grids and increments of the tests: every size the SCF accepts from 8 to 20 levels, log and uniform
LOG_GRIDS = [(8, 0.02, 10.0), (10, 0.004, 15.0), (11, 0.002, 15.0), (12, 0.001, 20.0), (13, 0.001, 15.0), (14, 0.0005, 25.0),
             (15, 0.0004, 50.0), (16, 0.0002, 50.0), (17, 1e-4, 50.0), (18, 5e-5, 50.0), (20, 1.25e-5, 50.0)]
UNIFORM_GRIDS = [(12, 0.0, 15.0), (14, 0.0, 15.0), (15, 0.0, 25.0)]
GRIDS = LOG_GRIDS + UNIFORM_GRIDS
CHUNK = 16384           # nodes per chunk of the direct solve above 14 levels (poisson_direct.cu)


def grid_r(L, delta, rmax):
    N = (1 << L) + 1
    if delta == 0.0:
        return np.arange(N) * (rmax / (N - 1))
    return O.grid(L, delta, rmax)[2]


def atom_density(Z, r):
    """A shell-like density of Z electrons: one exponential shell per row of the periodic table reached by Z."""
    rho = np.zeros_like(r)
    left, k = float(Z), 0.6 * Z
    for cap in (2, 8, 8, 18, 18, 32, 32):
        q = min(left, cap)
        rho += q * k ** 3 / np.pi * np.exp(-2.0 * k * r)
        left -= q
        k = max(0.35, k / 3.2)
        if left <= 0:
            break
    return rho


def increments(L, delta, rmax, seed=0):
    """(rho_prev, rho, labels) [8][N]: one density per kind of increment, Z from 1 to 92.  The increments: smooth shell-like changes of
    1e-2 .. 1e-9 of rho, rough node-by-node noise (every carry of the scans matters), changes confined to a few nodes at node 1, at node
    N-2 and on both sides of every chunk boundary 16384 k (on smaller grids: of N/4, N/2, 3N/4), and an all-zero increment."""
    r = grid_r(L, delta, rmax)
    N = len(r)
    rng = np.random.default_rng(seed + 31 * L)
    Zs = [1, 18, 54, 92, 36, 10, 86, 2]
    prev = np.stack([atom_density(Z, r) for Z in Zs])
    rho = prev.copy()
    x = r / r[-1]
    rho[0] = prev[0] * (1 + 1e-2 * np.cos(9.0 * x))
    rho[1] = prev[1] * (1 + 1e-5 * np.sin(25.0 * x) * np.exp(-3 * x))
    rho[2] = prev[2] * (1 + 1e-9 * np.cos(4.0 * np.sqrt(x)))
    rho[3] = prev[3] * (1 + 1e-6 * rng.standard_normal(N))
    rho[4, 1:4] += 1e-3 * rng.standard_normal(3) * max(prev[4, 1], 1.0)
    rho[5, N - 4:N - 1] += 1e-4 * rng.standard_normal(3)
    cuts = list(range(CHUNK, N - 1, CHUNK)) if N - 1 > CHUNK else [(N - 1) // 4, (N - 1) // 2, 3 * (N - 1) // 4]
    for c in cuts:
        rho[6, c - 2:c + 2] += 1e-6 * rng.standard_normal(4) * (1 + prev[6, c])
    rho[:, 0] = prev[:, 0]              # (node 0 and node N-1 carry no source: psrc = 0 there)
    labels = ["smooth 1e-2", "smooth 1e-5", "smooth 1e-9", "noise", "node 1", "node N-2", "chunk edges", "zero"]
    return prev, rho, labels
