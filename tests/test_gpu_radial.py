"""GPU tests of the radial export (Context.solve_batch(..., radial=True) / dftatom_solve_batch_radial): it changes nothing in the SCF,
returns the reference's own final fields (oracle orc_scf_ex), normalised orbitals with the right nodes, moments of the energies'
quadrature, the same arrays whatever the stream groups or the rest of the batch, and the same tables from the CLI."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import oracle_lib as O
from conftest import golden
from dftatom_b200.api import _COptions, _CRadial, _CResult

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FOUR_PI = 4.0 * np.pi


def _opt(o):
    return D.Options(o["Z"], o["levels"], o["rmax"], o["delta"], o["mixing"], o["method"])


def _grid(levels, delta, max_r):
    """r and the Simpson38-weighted jacobian of the engine's grid tables (engine.cpp get_grid)."""
    N = 2 ** levels + 1
    i = np.arange(N)
    w = np.where((i == 0) | (i == N - 1), 1.0, np.where(i % 3 == 0, 2.0, 3.0)) * 0.375
    if delta == 0.0:
        h = max_r / (N - 1)
        return max_r * i / (N - 1), w * h
    rp = max_r / (np.exp((N - 1) * delta) - 1.0)
    ex = np.exp(i * delta)
    return rp * (ex - 1.0), w * (rp * delta * ex)


def _grid_of(o):
    return _grid(o.MultigridLevels, 0.0 if o.method >= 2 else o.deltaGrid, o.MaxR)


def _sign_changes(u):
    s = np.sign(u[u != 0.0])
    return int(np.count_nonzero(s[1:] != s[:-1]))


def _records(res):
    return [(r.status, r.n_steps, [(s.E, s.Etotal, s.Ekin, s.Ecoul, s.Eenuc, s.Exc, s.levels_converged, s.stop_criterion_met) for s in r.steps])
            for r in res]


def _fields(res):
    out = []
    for r in res:
        x = r.radial
        out.append([x.r, x.rho, x.V, x.V_H, x.n_electrons, x.r2] + list(x.orbitals) + list(x.moments))
    return out


def _assert_same_fields(fa, fb):
    assert len(fa) == len(fb)
    for a, b in zip(fa, fb):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            assert np.array_equal(np.asarray(x), np.asarray(y))


def _check_orbitals(r, tol=1e-12):
    """unit norm with the Simpson38 jacobian, n - l - 1 sign changes, positive at the first non-zero node, node 0 = 0"""
    _, wj = _grid_of(r.options)
    x = r.radial
    for s, chan in enumerate(r.levels):
        assert x.orbitals[s].shape == (len(chan), len(wj))
        for k, L in enumerate(chan):
            u = x.orbitals[s][k]
            assert np.all(np.isfinite(u))
            assert abs(np.sum(wj * u * u) - 1.0) < tol, (r.options.Z, s, L.n, L.l)
            assert _sign_changes(u) == L.n - L.l - 1, (r.options.Z, s, L.n, L.l)
            assert u[0] == 0.0 and u[np.flatnonzero(u[1:])[0] + 1] > 0.0


def test_opt_in_changes_nothing(ctx):
    small = [_opt(a["options"]) for a in golden("small")["atoms"] if a["options"]["levels"] == 10]
    forty = [D.Options(Z, 12, 15.0, 0.001, 0.5, Z % 2) for Z in range(1, 41)]
    for opts in (small, forty):
        first = ctx.solve_batch(opts)       # the first solve on a grid also solves its start potential once (unit_guess): one launch more
        plain = ctx.solve_batch(opts)
        launches = ctx.last_timing()[1]
        _, d2h = ctx.last_transfer()
        rad = ctx.solve_batch(opts, radial=True)
        assert _records(first) == _records(plain) == _records(rad)
        assert all(r.radial is None for r in plain)
        assert ctx.last_timing()[1] == launches
        assert ctx.last_transfer()[1] > d2h


def _orc_scf_ex(o):
    L = O.oracle()
    L.orc_scf_ex.argtypes = [C.POINTER(O.OrcOptions), C.POINTER(O.OrcResult), O.STEP_CB, C.c_void_p, C.c_int, O._dp, O._dp]
    N = 2 ** o.MultigridLevels + 1
    V = np.zeros(2 * N)
    rho = np.zeros(2 * N)
    res = O.OrcResult()
    cb = O.STEP_CB(lambda st, user: None)
    L.orc_scf_ex(C.byref(O.OrcOptions(o.Z, o.MultigridLevels, o.MaxR, o.deltaGrid, o.alpha, o.method)), C.byref(res), cb, None, 100,
                 O.d(V), O.d(rho))
    return V.reshape(2, N), rho.reshape(2, N), res


@pytest.mark.parametrize("which", ["argon", "lsda"])
def test_fields_match_the_reference_fields(ctx, which):
    if which == "argon":
        o = _opt(golden("argon")["atoms"][0]["options"])
    else:
        o = next(_opt(a["options"]) for a in golden("small")["atoms"] if a["options"]["method"] == 1 and a["options"]["levels"] == 10)
    r = ctx.solve_batch([o], radial=True)[0]
    assert r.finished
    V_ref, rho_ref, ores = _orc_scf_ex(o)
    assert ores.finished
    x = r.radial
    rr, _ = _grid_of(o)
    np.testing.assert_allclose(x.r, rr, rtol=1e-12, atol=0)      # (libm's exp against numpy's)
    assert x.rho[:, 0].tolist() == [0.0] * len(x.rho) and x.V[:, 0].tolist() == [0.0] * len(x.V) and x.V_H[0] == 0.0
    ns = len(x.rho)
    q = FOUR_PI * rr * rr
    for s in range(ns):
        np.testing.assert_allclose(q * x.rho[s], q * rho_ref[s], rtol=0, atol=1e-6)
    mask = q * x.rho.sum(axis=0) > 1e-8
    for s in range(ns):
        np.testing.assert_allclose((rr * x.V[s])[mask], (rr * V_ref[s])[mask], rtol=0, atol=1e-6 * o.Z)
    # orbitals against the oracle's matched solution in the reference's final potential, at this run's eigenvalues
    _check_orbitals(r)
    for s, chan in enumerate(r.levels):
        for k, L in enumerate(chan):
            u_ref, _ = O.orbital(V_ref[s], o.deltaGrid, o.MaxR, L.l, L.E)
            u = x.orbitals[s][k]
            u_ref = u_ref * np.sign(u_ref[np.flatnonzero(u_ref[1:])[0] + 1])
            assert np.max(np.abs(u - u_ref)) <= 1e-6 * np.max(np.abs(u)), (o.Z, s, L.n, L.l)


def test_sweep_orbitals_density_and_moments(ctx):
    """C3 (Z = 1..92, LDA, 16385 nodes): every orbital normalised with the right nodes; the density rebuilt from the orbitals; moments
    equal to a numpy Simpson38 of the returned orbitals; electron count = Z.
    The density is mixed linearly from the uniform start density rho_0 = Z / volume (DFTAtom.cpp:371-376, :332-342): after n steps it
    still holds alpha^n rho_0 (4 pi r^2 alpha^n rho_0 ~ 1e-6 near Rmax after ~25 steps at alpha = 0.5), which no orbital carries.  That
    part is taken out before the comparison.  What remains is the SCF residual at the stop: the stop test is on the energy, which is
    stationary in the density, so it does not bound the density residual to first order.  Measured on a B200: <= 1e-6 in 4 pi r^2 rho
    for every finished atom of the sweep but Z = 90 (1.9e-6, its 5f / 6d shells still settle when the energy has converged)."""
    opts = [D.Options(Z, 14, 25.0, 0.0005, 0.5, 0) for Z in range(1, 93)]
    res = ctx.solve_batch(opts, keep_steps=False, radial=True)
    rr, wj = _grid(14, 0.0005, 25.0)
    q = FOUR_PI * rr * rr
    inv_r = np.zeros_like(rr)
    inv_r[1:] = 1.0 / rr[1:]
    for r in res:
        _check_orbitals(r)
        x = r.radial
        assert abs(x.n_electrons - r.options.Z) < 1e-8, (r.options.Z, x.n_electrons)
        assert abs(x.r2 - np.sum(wj * q * x.rho[0] * rr * rr)) <= 1e-12 * x.r2
        u = x.orbitals[0]
        for f, col in ((inv_r, 0), (rr, 1), (rr * rr, 2)):
            np.testing.assert_allclose(x.moments[0][:, col], (wj * f * u * u).sum(axis=1), rtol=1e-12, atol=0)
        if r.finished:
            occ = np.array([L.occ for L in r.levels[0]], dtype=np.float64)
            dens = (occ[:, None] * u * u).sum(axis=0)
            start = 0.5 ** r.n_steps * r.options.Z / (FOUR_PI / 3.0 * 25.0 ** 3)
            np.testing.assert_allclose(dens[1:-1], (q * (x.rho[0] - start))[1:-1], rtol=0, atol=2e-6 if r.options.Z == 90 else 1e-6,
                                       err_msg=f"Z={r.options.Z}")


def test_radial_moments_of_hydrogenic_orbitals(ctx):
    levels, delta, max_r = 14, 0.0008, 60.0
    rr, _ = _grid(levels, delta, max_r)
    for Z in (1.0, 3.0):
        V = np.zeros_like(rr)
        V[1:] = -Z / rr[1:]
        rows, want = [], []
        for n, l, m in ((1, 0, (Z, 1.5 / Z, 3.0 / Z ** 2)), (2, 1, (Z / 4.0, 5.0 / Z, 30.0 / Z ** 2))):
            u, _ = ctx.numerov_orbital(V, levels, delta, max_r, l, -Z * Z / (2.0 * n * n))
            rows.append(u)
            want.append(m)
        got = ctx.radial_moments(levels, delta, max_r, np.array(rows))
        np.testing.assert_allclose(got, np.array(want), rtol=1e-6, atol=0)


def test_stream_groups_scatter_the_same_fields():
    opts = [D.Options(Z, 12, 15.0, 0.001, 0.5, (Z // 3) % 2) for Z in range(1, 41)]
    out = []
    for groups in (4, 1):
        with D.Context(0) as c:
            c.set_option("stream_groups", groups)
            out.append(c.solve_batch(opts, keep_steps=False, radial=True))
    _assert_same_fields(_fields(out[0]), _fields(out[1]))
    assert [r.options.Z for r in out[0]] == list(range(1, 41))


def test_finished_atom_keeps_its_fields(ctx):
    """Z = 2 stops long before Z = 68..70: its arrays are frozen at its own last step, equal to Z = 2 solved alone."""
    mk = lambda Z: D.Options(Z, 12, 15.0, 0.001, 0.5, 0)
    mixed = ctx.solve_batch([mk(68), mk(2), mk(69), mk(70)], radial=True)
    alone = ctx.solve_batch([mk(2)], radial=True)
    assert mixed[1].n_steps < max(r.n_steps for r in mixed)
    _assert_same_fields(_fields([mixed[1]]), _fields(alone))


def test_large_grid_and_uniform_paths(ctx):
    """65537 nodes (stream-mode Poisson, padded U rows) and the uniform grid: finite fields, unit-norm orbitals, right node counts."""
    lsda = [_opt(a["options"]) for a in golden("lsda_batch")["atoms"]]
    uni = [_opt(a["options"]) for a in golden("uniform")["atoms"] if a["options"]["levels"] == 12]
    for opts in (lsda, uni):
        for r in ctx.solve_batch(opts, keep_steps=False, radial=True):
            x = r.radial
            assert all(np.all(np.isfinite(a)) for a in (x.rho, x.V, x.V_H))
            assert abs(x.n_electrons - r.options.Z) < 1e-6 * r.options.Z
            _check_orbitals(r, tol=1e-11)


def test_too_few_orbital_rows_is_an_argument_error(ctx):
    lib = D.load_library()
    opts = [D.Options(18, 10, 15.0, 0.004, 0.5, 0), D.Options(7, 10, 15.0, 0.004, 0.5, 1)]
    rows = D.orbital_count(18, 0) + D.orbital_count(7, 1)
    N = D.n_nodes(10)
    orb = np.zeros((rows, N))
    copts = (_COptions * 2)(*[o._c() for o in opts])
    cres = (_CResult * 2)()
    rad = _CRadial(None, None, None, None, orb.ctypes.data_as(C.POINTER(C.c_double)), rows - 1, None, None)
    assert lib.dftatom_solve_batch_radial(ctx._h, copts, 2, cres, None, 0, C.byref(rad)) == -5        # DFTATOM_E_ARG
    assert not orb.any()
    rad.orbital_rows = rows
    assert lib.dftatom_solve_batch_radial(ctx._h, copts, 2, cres, None, 0, C.byref(rad)) == 0
    assert orb.any()


def _run_cli(args, tmp):
    exe = os.path.join(ROOT, "bin", "dftatom")
    subprocess.run([exe] + args + ["--radial", tmp, "--quiet-steps"], check=True, capture_output=True, text=True)
    return {f: np.loadtxt(os.path.join(tmp, f), delimiter="\t", ndmin=2) for f in sorted(os.listdir(tmp))}


def test_cli_writes_the_python_arrays(ctx):
    zs = [10, 18, 3]
    opts = [D.Options(Z, 12, 15.0, 0.001, 0.5, 1) for Z in zs]
    res = ctx.solve_batch(opts, radial=True)
    args = ["--Z", ",".join(map(str, zs)), "--levels", "12", "--delta", "0.001", "--rmax", "15", "--mixing", "0.5", "--method", "1"]
    with tempfile.TemporaryDirectory() as tmp:
        tabs = _run_cli(args, tmp)
        with open(os.path.join(tmp, "1_Z18.tsv")) as fh:
            head = fh.readline().rstrip("\n").split("\t")
    assert sorted(tabs) == [f"{i}_Z{Z}.tsv" for i, Z in enumerate(zs)]
    assert head[:6] == ["# r", "rho alpha", "rho beta", "V alpha", "V beta", "V_H"] and head[6] == "alpha 1s"
    for i, r in enumerate(res):
        x = r.radial
        want = np.column_stack([x.r] + list(x.rho) + list(x.V) + [x.V_H] + [u for ch in x.orbitals for u in ch])
        assert np.array_equal(tabs[f"{i}_Z{zs[i]}.tsv"], want)
    import torch
    if torch.cuda.device_count() >= 2:
        with tempfile.TemporaryDirectory() as tmp:
            tabs2 = _run_cli(args + ["--gpus", "2"], tmp)
        assert sorted(tabs2) == sorted(tabs)
        for f in tabs:
            assert np.array_equal(tabs2[f], tabs[f])
