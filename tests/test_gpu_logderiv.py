"""GPU tests of the logarithmic derivatives (Context.log_derivatives / dftatom_log_derivatives): parity with the numpy reference of
tests/logderiv_ref.py on converged potentials of both grids and both spins, the hydrogen atom, the monotone phase, the Wronskian
identity, the node counts at the eigenvalues, independence of the batch, overflow, argument validation and the CLI tables."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import logderiv_ref as R
from dftatom_b200.api import _CLogDeriv

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AR = D.Options(18, 14, 25.0, 0.0005, 0.5, 0)        # C1


def _grid_args(o):
    return o.MultigridLevels, 0.0 if o.method >= 2 else o.deltaGrid, o.MaxR


_solved = {}


def _radial(ctx, o):
    """The converged radial state of one atom (Result.radial), solved once per session."""
    key = (o.Z, o.MultigridLevels, o.MaxR, o.deltaGrid, o.method)
    if key not in _solved:
        _solved[key] = ctx.solve_batch([o], keep_steps=False, radial=True)[0]
    return _solved[key].radial


def _V(ctx, o):
    return _radial(ctx, o).V


def _assert_parity(got, ch, V, grid, l, r_c, E):
    Dr, ur, dur, nr, rr = R.log_derivative(V, *grid, l, r_c, E)
    assert abs(got.r_c[ch] - rr) <= 1e-14 * rr                       # the same node (the radii may differ in the last bit: libm)
    assert np.array_equal(got.nodes[ch], nr)
    ok = np.abs(rr * Dr) < 1e3
    assert ok.sum() > len(E) // 2
    # relative to the scale of the pair (u, r_c u'), which stays away from zero where u crosses it
    scale = np.hypot(ur, rr * dur)[ok]
    assert np.all(np.abs(got.D[ch][ok] - Dr[ok]) <= 1e-9 * np.maximum(np.abs(Dr[ok]), 1.0 / rr))
    assert np.all(np.abs(got.u[ch][ok] - ur[ok]) <= 1e-9 * scale)
    assert np.all(np.abs(got.du[ch][ok] - dur[ok]) * rr <= 1e-9 * scale)


def test_parity_with_the_reference_on_hydrogen(ctx):
    grid = (12, 0.002, 25.0)
    N, r, _, _ = R.grid(*grid)
    V = np.zeros(N)
    V[1:] = -1.0 / r[1:]
    E = np.linspace(-3.0, 5.0, 97)
    got = ctx.log_derivatives(V, *grid, 0, [0, 1, 2, 3], 2.0, E)
    for l in range(4):
        _assert_parity(got, l, V, grid, l, 2.0, E)


@pytest.mark.parametrize("o,r_c", [(AR, 2.5), (D.Options(26, 14, 25.0, 0.0005, 0.5, 1), 2.2), (D.Options(10, 14, 15.0, 0.0005, 0.5, 2), 1.7)],
                         ids=["Ar-LDA", "Fe-LSDA", "Ne-uniform"])
def test_parity_with_the_reference_on_converged_potentials(ctx, o, r_c):
    V = _V(ctx, o)
    grid = _grid_args(o)
    E = np.concatenate([np.linspace(-3.0, 3.0, 61), [-120.0, -10.5, -0.3]])
    pot = [s for s in range(len(V)) for _ in range(4)][::-1]        # LSDA: beta rows first, so a swapped row index shows
    l = [k % 4 for k in range(len(pot))]
    got = ctx.log_derivatives(V, *grid, pot, l, r_c, E)
    for ch in range(len(pot)):
        _assert_parity(got, ch, V[pot[ch]], grid, l[ch], r_c, E)


def test_parity_on_radon_lsda_at_131073_nodes(ctx):
    o = D.Options(86, 17, 50.0, 0.0001, 0.5, 1)                    # C2
    V = _V(ctx, o)
    grid = _grid_args(o)
    E = np.array([-3.0, -0.5, 0.7])
    got = ctx.log_derivatives(V, *grid, [0, 1], [0, 3], 1.8, E)
    _assert_parity(got, 0, V[0], grid, 0, 1.8, E)
    _assert_parity(got, 1, V[1], grid, 3, 1.8, E)


def test_hydrogen_analytic_values(ctx):
    grid = (14, 0.0005, 25.0)
    N, r, _, _ = R.grid(*grid)
    V = np.zeros(N)
    V[1:] = -1.0 / r[1:]
    a = ctx.log_derivatives(V, *grid, 0, 0, 2.0, [-0.5])
    b = ctx.log_derivatives(V, *grid, 0, 1, 2.0, [-0.125])
    rc = a.r_c[0]
    i0 = 0.25 - np.exp(-2 * rc) * (rc * rc / 2 + rc / 2 + 0.25)
    i1 = 24 - np.exp(-rc) * (rc ** 4 + 4 * rc ** 3 + 12 * rc ** 2 + 24 * rc + 24)
    assert abs(a.D[0, 0] - (1 / rc - 1)) < 1e-8 and abs(b.D[0, 0] - (2 / rc - 0.5)) < 1e-8
    assert abs(a.u[0, 0] - rc * np.exp(-rc) / np.sqrt(i0)) < 1e-8
    assert abs(b.u[0, 0] - rc * rc * np.exp(-rc / 2) / np.sqrt(i1)) < 1e-8
    assert a.nodes[0, 0] == 0 and b.nodes[0, 0] == 0


def test_phase_is_strictly_increasing_through_the_bound_levels_of_argon(ctx):
    V = _V(ctx, AR)
    E = np.linspace(-120.0, 5.0, 2501)                              # 1s at -113.8 Ha up into the continuum
    got = ctx.log_derivatives(V, *_grid_args(AR), 0, [0, 1, 2, 3], 2.0, E)
    assert np.all(got.nodes >= 0) and np.all(np.isfinite(got.D))
    assert np.all(np.diff(got.phase, axis=1) > 0)
    assert got.nodes[0, -1] >= 3 and got.nodes[1, -1] >= 2          # 1s 2s 3s / 2p 3p are below 5 Ha


def test_wronskian_identity(ctx):
    V = _V(ctx, AR)
    E = np.linspace(-2.0, 2.0, 201)
    h = 1e-5
    args = (V, *_grid_args(AR), 0, [0, 1, 2, 3], 2.0)
    got = ctx.log_derivatives(*args, E)
    dD = (ctx.log_derivatives(*args, E + h).D - ctx.log_derivatives(*args, E - h).D) / (2 * h)
    ok = np.abs(got.r_c[:, None] * got.D) < 20
    assert ok.sum() > 400
    assert np.max(np.abs(-0.5 * dD[ok] * got.u[ok] ** 2 - 1.0)) < 1e-5


def test_node_counts_bracket_the_eigenvalues(ctx):
    V = _V(ctx, AR)
    levels, delta, max_r = _grid_args(AR)
    ns, ls = [1, 2, 2, 3, 3], [0, 0, 1, 0, 1]
    eps, ok = ctx.level_search(V[0], levels, delta, max_r, 18, ns, ls)
    assert ok.all()
    r_far = _radial(ctx, AR).r[-3]                                   # r_(N-2) of the engine's grid
    for n, l, e in zip(ns, ls, eps):
        de = max(1e-6, 1e-8 * abs(e))
        got = ctx.log_derivatives(V, levels, delta, max_r, 0, l, r_far, [e - de, e + de])
        assert got.r_c[0] == r_far
        assert got.nodes[0].tolist() == [n - l - 1, n - l], (n, l, e)


def test_channel_is_independent_of_the_batch(ctx):
    opts = [D.Options(Z, 14, 25.0, 0.0005, 0.5, 0) for Z in range(1, 93)]     # C3
    res = ctx.solve_batch(opts, keep_steps=False, radial=True)
    V = np.concatenate([r.radial.V for r in res])
    E = np.linspace(-2.0, 2.0, 301)
    grid = _grid_args(opts[0])
    pot = np.repeat(np.arange(92), 4)
    l = np.tile(np.arange(4), 92)
    r_c = np.where(pot % 3 == 0, 2.5, 1.5)                             # two sweep lengths: the warps are reordered
    batch = ctx.log_derivatives(V, *grid, pot, l, r_c, E)
    for ch in (0, 17 * 4 + 2, 91 * 4 + 3):
        alone = ctx.log_derivatives(V[pot[ch]], *grid, 0, l[ch], r_c[ch], E)
        for f in ("D", "u", "du", "nodes"):
            assert np.array_equal(getattr(alone, f)[0], getattr(batch, f)[ch], equal_nan=True), (ch, f)
        assert alone.r_c[0] == batch.r_c[ch]


def test_deep_energy_at_the_outermost_radius_stays_finite(ctx):
    o = D.Options(86, 17, 50.0, 0.0001, 0.5, 1)
    V = _V(ctx, o)
    levels, delta, max_r = _grid_args(o)
    r_far = _radial(ctx, o).r[-3]
    got = ctx.log_derivatives(V, levels, delta, max_r, [0, 1, 0, 1], [0, 0, 3, 3], r_far, [-86.0 ** 2 - 1, -5.0, 2.0])
    assert np.all(got.nodes >= 0)
    for f in (got.D, got.u, got.du):
        assert np.all(np.isfinite(f))
    assert np.all(got.D[:, 0] > 0)                                    # far below every level: the solution grows


def test_invalid_arguments_are_rejected_before_any_launch(ctx):
    lib = D.load_library()
    levels, delta, max_r = 12, 0.002, 25.0
    N, r, _, _ = R.grid(levels, delta, max_r)
    V = np.zeros((2, N))
    V[:, 1:] = -1.0 / r[1:]

    def call(V=V, n_pot=2, pot=(0,), l=(0,), r_c=(2.0,), E=(-0.5,), n_ch=None, n_e=None, grid=(levels, delta, max_r)):
        V = np.ascontiguousarray(V, dtype=np.float64)
        pot = np.array(pot, np.int32); l = np.array(l, np.int32); r_c = np.array(r_c, np.float64); E = np.array(E, np.float64)
        n_ch = len(pot) if n_ch is None else n_ch
        n_e = len(E) if n_e is None else n_e
        out = np.full(max(1, len(pot) * len(E)), 7.0, dtype=np.dtype(_CLogDeriv))
        used = np.full(max(1, len(pot)), 7.0)
        rc = lib.dftatom_log_derivatives(ctx._h, grid[0], grid[1], grid[2], V.ctypes.data_as(C.POINTER(C.c_double)), n_pot,
                                         pot.ctypes.data_as(C.POINTER(C.c_int)), l.ctypes.data_as(C.POINTER(C.c_int)),
                                         r_c.ctypes.data_as(C.POINTER(C.c_double)), n_ch, E.ctypes.data_as(C.POINTER(C.c_double)), n_e,
                                         out.ctypes.data_as(C.POINTER(_CLogDeriv)), used.ctypes.data_as(C.POINTER(C.c_double)))
        untouched = bool(np.all(out["D"] == 7.0) and np.all(used == 7.0))
        return rc, lib.dftatom_last_error().decode(), untouched

    rc, _, _ = call()
    assert rc == 0
    bad_V = V.copy()
    bad_V[1, 5] = np.nan
    cases = [
        (dict(grid=(0, delta, max_r)), -2, "grid"),
        (dict(grid=(levels, -1.0, max_r)), -2, "grid"),
        (dict(n_pot=0), -5, ""),
        (dict(n_ch=0), -5, ""),
        (dict(n_e=0), -5, ""),
        (dict(pot=(0, 2), l=(0, 0), r_c=(2.0, 2.0)), -5, "channel 1"),
        (dict(pot=(-1,)), -5, "channel 0"),
        (dict(l=(4,)), -5, "channel 0"),
        (dict(l=(-1,)), -5, "channel 0"),
        (dict(r_c=(0.5 * r[2],)), -5, "channel 0"),
        (dict(r_c=(r[N - 2] * 1.0001,)), -5, "channel 0"),
        (dict(r_c=(np.nan,)), -5, "channel 0"),
        (dict(E=(-0.5, np.inf)), -5, "energy 1"),
        (dict(E=(np.nan,)), -5, "energy 0"),
        (dict(V=bad_V), -5, "potential row 1"),
    ]
    for kw, code, text in cases:
        rc, msg, untouched = call(**kw)
        assert rc == code, (kw, rc, msg)
        assert text in msg, (kw, msg)
        assert untouched, kw
    with pytest.raises(D.DFTAtomError, match="error -5"):
        ctx.log_derivatives(V, levels, delta, max_r, 0, 5, 2.0, [-0.5])
    # the bounds themselves are valid: r_2 and r_(N-2) as the engine returns them
    ends = ctx.log_derivatives(V, levels, delta, max_r, 0, 0, [r[2] * (1 + 1e-9), r[N - 2] * (1 - 1e-9)], [-0.5]).r_c
    assert np.allclose(ends, [r[2], r[N - 2]], rtol=1e-14, atol=0)
    assert ctx.log_derivatives(V, levels, delta, max_r, 0, 0, ends, [-0.5]).r_c.tolist() == ends.tolist()


def _run_cli(args):
    exe = os.path.join(ROOT, "bin", "dftatom")
    with tempfile.TemporaryDirectory() as tmp:
        ld, rad = os.path.join(tmp, "ld"), os.path.join(tmp, "rad")
        subprocess.run([exe] + args + ["--logderiv", ld, "--radial", rad, "--quiet-steps"], check=True, capture_output=True, text=True)
        tabs = {f: open(os.path.join(ld, f)).read() for f in sorted(os.listdir(ld))}
        V = {f: np.loadtxt(os.path.join(rad, f), delimiter="\t", ndmin=2) for f in sorted(os.listdir(rad))}
    return tabs, V


def test_cli_writes_what_the_python_call_returns(ctx):
    args = ["--Z", "18", "--rc", "2", "--energies", "-2:1:31"]
    tabs, rad = _run_cli(args)
    assert sorted(tabs) == ["0_Z18_logderiv.tsv"]
    lines = tabs["0_Z18_logderiv.tsv"].splitlines()
    assert lines[0].startswith("# Z=18 method=0 r_c=")
    assert lines[1] == "# spin\tl\tE\tD\tnodes\tphase\tu\tdu"
    t = np.loadtxt(lines[2:], delimiter="\t", ndmin=2)
    assert t.shape == (4 * 31, 8)
    E = t[:31, 2]
    assert E[0] == -2.0 and E[-1] == 1.0
    V = rad["0_Z18.tsv"][:, 2]                                      # columns r | rho | V | V_H | orbitals
    got = ctx.log_derivatives(V, 12, 0.001, 10.0, 0, [0, 1, 2, 3], 2.0, E)   # the CLI's default grid (Options.cpp)
    assert float(lines[0].split("r_c=")[1]) == got.r_c[0]
    for l in range(4):
        blk = t[31 * l:31 * (l + 1)]
        assert np.all(blk[:, 0] == 0) and np.all(blk[:, 1] == l) and np.array_equal(blk[:, 2], E)
        assert np.array_equal(blk[:, 3], got.D[l]) and np.array_equal(blk[:, 4], got.nodes[l])
        assert np.array_equal(blk[:, 6], got.u[l]) and np.array_equal(blk[:, 7], got.du[l])
        assert np.allclose(blk[:, 5], got.phase[l], rtol=1e-15, atol=1e-14)
    import torch
    if torch.cuda.device_count() >= 2:
        multi = ["--Z", "3,18,10", "--method", "1", "--rc", "1.5", "--energies", "-1:1:40"]
        one, _ = _run_cli(multi)
        two, _ = _run_cli(multi + ["--gpus", "2"])
        assert sorted(one) == ["0_Z3_logderiv.tsv", "1_Z18_logderiv.tsv", "2_Z10_logderiv.tsv"]
        assert one == two
