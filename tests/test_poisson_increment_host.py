"""CPU self-checks of tests/poisson_increment_ref.py, the exact solution of the warm Poisson solves' linear system that
tests/test_gpu_poisson_increment.py measures the kernels against."""
import numpy as np
import pytest

import poisson_increment_ref as R
from poisson_increment_ref import GRIDS, LOG_GRIDS


@pytest.mark.parametrize("delta", [0.02, 0.0])
def test_reference_equals_exact_rationals(delta):
    """8 levels (257 nodes): the __float128 solve, rounded once, is the exact rational solution rounded (within 1 ulp of the largest)."""
    rng = np.random.default_rng(5)
    N = 257
    for h in (rng.standard_normal(N), np.exp(-np.linspace(0, 8, N)) * 1e-3, np.where(np.arange(N) == 1, 1.0, 0.0)):
        got = R.solve_h(delta, h)
        exact = R.solve_fraction(delta, h)
        scale = max(abs(float(x)) for x in exact)
        err = max(abs(float(x - type(x)(g))) for x, g in zip(exact, got))
        assert err <= 2.3e-16 * scale, (err, scale)
        assert got[0] == 0.0 and got[-1] == 0.0


@pytest.mark.parametrize("L,delta,rmax", GRIDS)
def test_reference_agrees_with_fp64_banded_solve(L, delta, rmax):
    """Every grid of the GPU tests, on their increments: scipy's FP64 banded solve (LU with partial pivoting) lands within FP64's
    expected error of the reference, which grows with the condition of the system, ~N^2: measured 1e-3 eps N^2 at every size (1.6e-7
    relative at 1048577 nodes, 1.5e-14 at 257), bound 4e-3 eps N^2.  The residual of the reference in the FP64 system is at the
    rounding level of its terms."""
    prev, rho, _ = R.increments(L, delta, rmax)
    N = rho.shape[1]
    ex = R.solve(L, delta, rmax, rho, prev)
    a, b = R.coefficients(delta)
    for k in range(rho.shape[0] - 1):
        h = R.rhs(L, delta, rmax, rho[k], prev[k])
        fp = R.solve_banded_fp64(delta, h)
        scale = np.max(np.abs(ex[k]))
        assert scale > 0
        assert np.max(np.abs(fp - ex[k])) <= 4e-3 * 2.2e-16 * float(N) ** 2 * scale, (k, np.max(np.abs(fp - ex[k])) / scale)
        res = -a * ex[k][:-2] + ex[k][1:-1] - b * ex[k][2:] - h[1:-1]
        terms = np.abs(a * ex[k][:-2]) + np.abs(ex[k][1:-1]) + np.abs(b * ex[k][2:]) + np.abs(h[1:-1])
        assert np.all(np.abs(res) <= 4 * 2.2e-16 * terms), k
    assert np.all(ex[-1] == 0.0)                # the zero increment


def test_reference_builds_the_engines_source_factor():
    """psrc_i = r_i 4 pi K_i with the grid of the oracle (and the engine): r from O.grid, K = (rp delta)^2 e^{2 delta i}."""
    import oracle_lib as O
    for L, delta, rmax in LOG_GRIDS[:4]:
        _, rp, r = O.grid(L, delta, rmax)
        i = np.arange(len(r))
        ref = r * (4 * np.pi * rp * rp * delta * delta * np.exp(2 * delta * i))
        ref[0] = ref[-1] = 0.0
        np.testing.assert_allclose(R.psrc(L, delta, rmax), ref, rtol=1e-12, atol=0)
