"""GPU tests of the self-consistent pseudo-atom (Context.solve_pseudo_batch / dftatom_solve_pseudo_batch) on C, Si and Cu pseudized as in
tests/test_gpu_pseudo.py: the reference configuration against the all-electron atom the pseudopotential came from, parity with the
numpy reference of tests/pseudo_scf_ref.py (LDA and LSDA), LSDA with equal spins against LDA, the transferability test against the
all-electron atom in other configurations, independence of the batch, argument validation and the CLI table."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import pseudo_scf_ref as PS
from dftatom_b200.api import _CConfig, _COccupation, _CPseudoAtom, _CRadial, _CResult

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATOMS = {
    "C": (D.Options(6, 14, 25.0, 0.0005, 0.5, 0), 1.8, "[He]"),
    "Si": (D.Options(14, 14, 25.0, 0.0005, 0.5, 0, config="[Ne] 3s2 3p2 3d0"), 2.2, "[Ne]"),
    "Cu": (D.Options(29, 14, 25.0, 0.0005, 0.5, 0, config="[Ar] 3d10 4s1 4p0"), 2.2, "[Ar]"),
}
ADAPTIVE = {"Cu"}       # the fixed linear mixing does not settle Cu's nearly full 3d shell in 100 steps (all-electron and pseudo)
# (atom, valence configuration): the excitations of the transferability test, against the reference configuration of the atom
EXCITED = [("Si", "3s1 3p3"), ("Si", "3s2 3p1"), ("C", "2s1 2p3"), ("Cu", "3d9 4s2")]

_solved = {}


def _adaptive(ctx, name):
    ctx.set_option("adaptive_mixing", int(name in ADAPTIVE))


def _pp(ctx, name):
    if name not in _solved:
        o, r_c, _ = ATOMS[name]
        _adaptive(ctx, name)
        try:
            res = ctx.solve_batch([o], keep_steps=False, radial=True)[0]
        finally:
            ctx.set_option("adaptive_mixing", 0)
        assert res.finished
        pp = ctx.pseudize(res, r_c)
        assert np.all(pp.status == 0)
        _solved[name] = (o, res, pp)
    return _solved[name]


def _ref_valence(pp):
    return " ".join(f"{n}{'spdf'[l]}{occ:g}" for n, l, occ in sorted(zip(pp.n.tolist(), pp.l.tolist(), pp.occ.tolist())))


def _solve_ps(ctx, name, configs, **kw):
    _adaptive(ctx, name)
    try:
        return ctx.solve_pseudo_batch(_pp(ctx, name)[2], configs, **kw)
    finally:
        ctx.set_option("adaptive_mixing", 0)


def _solve_ae(ctx, name, valence):
    o, _, core = ATOMS[name]
    opts = [D.Options(o.Z, o.MultigridLevels, o.MaxR, o.deltaGrid, o.alpha, o.method, config=f"{core} {v}") for v in valence]
    _adaptive(ctx, name)
    try:
        return ctx.solve_batch(opts, keep_steps=False)
    finally:
        ctx.set_option("adaptive_mixing", 0)


@pytest.fixture(scope="module")
def ctx():
    with D.Context(0) as c:
        yield c


# measured on a B200 (max over C, Si, Cu): |eps_PS - eps_AE| 2.6e-6 Ha (Si, with its empty 3d box state; C 7.5e-10, Cu 3.0e-8), tolerance
# 7.5e-6.  Beyond r_c: orbitals 5.2e-5, density 1.0e-10 bohr^-3; V_ion + v - V_scr 3.9e-5 Ha over nodes 1..N-1 (tolerances 1.5e-4, 3e-10,
# 1.2e-4: 3x the measured maxima)
EPS_TOL, U_TOL, RHO_TOL, V_TOL = 7.5e-6, 1.5e-4, 3e-10, 1.2e-4


@pytest.mark.parametrize("name", sorted(ATOMS))
def test_reference_configuration_reproduces_the_all_electron_atom(ctx, name):
    o, res, pp = _pp(ctx, name)
    r = _solve_ps(ctx, name, _ref_valence(pp), radial=True)[0]
    assert r.finished, r.status
    N = len(pp.r)
    lev = {(L.n, L.l): (k, L) for k, L in enumerate(r.levels[0])}
    errs = {}
    for c, (l, n) in enumerate(zip(pp.l.tolist(), pp.n.tolist())):
        k, L = lev[(n, l)]
        assert L.nodes == 0
        errs.setdefault("eps", []).append(abs(L.E - pp.eps[c]))
        ic = int(np.searchsorted(pp.r, pp.r_c[c]))
        errs.setdefault("u", []).append(np.max(np.abs(r.radial.orbitals[0][k][ic + 1:] - pp.u[c][ic + 1:])))
        errs.setdefault("V", []).append(np.max(np.abs(pp.V_ion[c][1:] + r.radial.V[0][1:] - pp.V_scr[c][1:])))
    ic = int(np.searchsorted(pp.r, np.max(pp.r_c)))
    errs["rho"] = [np.max(np.abs(r.radial.rho[0][ic + 1:N - 1] - pp.rho_val[0][ic + 1:N - 1]))]
    print(f"MEASURED reference {name}: " + " ".join(f"{k} {max(v):.3e}" for k, v in errs.items()))
    assert max(errs["eps"]) <= EPS_TOL
    assert max(errs["u"]) <= U_TOL
    assert max(errs["rho"]) <= RHO_TOL
    assert max(errs["V"]) <= V_TOL
    assert abs(r.Ekin + r.Eenuc + r.Ecoul + r.Exc - r.Etotal) < 1e-8


# measured on a B200 (max over the cases): eigenvalues 1.5e-9 Ha, energies 5.3e-9 Ha (Si with an empty 3d entry: 1.1e-6 Ha on the unbound
# 3d box state, whose eigenvalue follows the density tail; the case solves 3s and 3p only)
@pytest.mark.parametrize("name,config,method", [("C", "2s2 2p2", 0), ("C", "2s1 2p3", 0), ("Si", "3s1 3p3", 0), ("C", "2s1/1 2p2/0", 1)])
def test_parity_with_the_numpy_reference(ctx, name, config, method):
    o, _, pp = _pp(ctx, name)
    r = _solve_ps(ctx, name, config, method=method)[0]
    assert r.finished
    v_ion = {int(l): pp.V_ion[c] for c, l in enumerate(pp.l.tolist())}
    n_ref = {int(l): int(n) for l, n in zip(pp.l.tolist(), pp.n.tolist())}
    entries = [e if len(e) == 4 else (e[0], e[1], 0, e[2]) for e in D.parse_config(config, method)]
    ref = PS.solve(v_ion, n_ref, entries, o.MultigridLevels, o.deltaGrid, o.MaxR, mixing=0.5, method=method)
    assert ref["converged"]
    de = max(abs(L.E - ref["E"][s][k]) for s, ch in enumerate(r.levels) for k, L in enumerate(ch))
    dE = max(abs(getattr(r, k) - ref[k]) for k in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"))
    print(f"MEASURED parity {name} {config} method {method}: eps {de:.3e} energies {dE:.3e} steps {r.n_steps} / {ref['n_steps']}")
    assert de < 1e-6
    assert dE < 1e-5


# measured on a B200: 1.7e-12 Ha on the eigenvalues, 2.0e-11 Ha on the energies; stated tolerance 1e-10 Ha
def test_lsda_with_equal_spins_equals_lda(ctx):
    lda = _solve_ps(ctx, "C", "2s2 2p2")[0]
    lsda = _solve_ps(ctx, "C", "2s1/1 2p1/1", method=1)[0]
    assert lda.finished and lsda.finished
    de = max(abs(a.E - b.E) for s in range(2) for a, b in zip(lda.levels[0], lsda.levels[s]))
    dE = max(abs(getattr(lda, k) - getattr(lsda, k)) for k in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"))
    print(f"MEASURED LSDA = LDA: eps {de:.3e} energies {dE:.3e}")
    assert de < 1e-10 and dE < 1e-10


def test_transferability_against_the_all_electron_atom(ctx):
    out = []
    for name, cfg in EXCITED:
        pp = _pp(ctx, name)[2]
        ref = _ref_valence(pp)
        extra = " 3d0" if name == "Si" else (" 4p0" if name == "Cu" else "")
        ps = _solve_ps(ctx, name, [ref, cfg + extra])
        ae = _solve_ae(ctx, name, [ref, cfg + extra])
        assert all(x.finished for x in ps + ae), [(x.status, x.n_steps) for x in ps + ae]
        d_ps, d_ae = ps[1].Etotal - ps[0].Etotal, ae[1].Etotal - ae[0].Etotal
        out.append((name, cfg, d_ae, d_ps))
    print("MEASURED transferability: " + "; ".join(f"{n} {c}: dE_AE {a:.6f} dE_PS {p:.6f} diff {p - a:+.2e}" for n, c, a, p in out))
    for n, c, a, p in out:
        assert abs(p - a) <= 1e-2, (n, c, a, p)


def test_a_pseudo_atom_is_independent_of_its_batch(ctx):
    pp_c, pp_si = _pp(ctx, "C")[2], _pp(ctx, "Si")[2]
    alone = ctx.solve_pseudo_batch(pp_c, "2s1 2p3")[0]
    pps = [pp_si if k % 2 else pp_c for k in range(201)]
    cfgs = ["3s2 3p2 3d0" if k % 2 else ("2s1 2p3" if k == 100 else "2s2 2p2") for k in range(201)]
    batch = ctx.solve_pseudo_batch(pps, cfgs)[100]
    assert alone.n_steps == batch.n_steps and alone.status == batch.status
    for k in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"):
        assert getattr(alone, k) == getattr(batch, k), k
    for a, b in zip(alone.steps, batch.steps):
        assert a == b
    assert [L.E for L in alone.levels[0]] == [L.E for L in batch.levels[0]]


def _raw(ctx, v_ion, atoms, configs, levels=14, delta=0.0005, max_r=25.0, radial=None):
    n = len(atoms)
    ca = (_CPseudoAtom * n)(*atoms)
    cc = (_CConfig * n)()
    for a, cfg in enumerate(configs):
        cc[a].n_orbitals = len(cfg)
        for k, e in enumerate(cfg):
            cc[a].orb[k] = _COccupation(*e)
    out = (_CResult * n)()
    C.memset(out, 0x5A, C.sizeof(out))
    V = np.ascontiguousarray(v_ion, np.float64)
    rc = ctx._lib.dftatom_solve_pseudo_batch(ctx._h, levels, delta, max_r, V.ctypes.data_as(C.POINTER(C.c_double)), V.shape[0], ca, cc, n, out,
                                             None, 0, radial)
    untouched = all(b == 0x5A for b in bytes(out))
    return rc, untouched


def test_invalid_arguments_are_rejected_before_any_launch(ctx):
    pp = _pp(ctx, "C")[2]
    V = pp.V_ion
    good = _CPseudoAtom((0, 1, -1, -1), (2, 2, 0, 0), 4.0, 0.5, 0, 0)
    cfg = [(2, 0, 0, 2.0), (2, 1, 0, 2.0)]
    rc, _ = _raw(ctx, V, [good], [cfg])
    assert rc == 0
    bad_v = V.copy(); bad_v[1, 77] = np.nan
    deep = V.copy(); deep[0, 5] = -2e4
    cases = [
        (dict(delta=0.0), [good], [cfg], V, -2),                                            # uniform grid
        ({}, [good], [[(2, 0, 0, 2.0), (3, 2, 0, 1.0)]], V, -2),                           # l without channel
        ({}, [good], [[(1, 0, 0, 2.0), (2, 1, 0, 2.0)]], V, -2),                           # n < n_ref
        ({}, [good], [[(2, 0, 0, 2.5), (2, 1, 0, 2.0)]], V, -2),                           # occupation above 2 (2l + 1)
        ({}, [good], [[(2, 0, 0, 2.0), (2, 0, 0, 1.0)]], V, -2),                           # duplicate entry
        ({}, [good], [[(2, 0, 0, 2.0), (2, 1, 0, 5.0)]], V, -2),                           # Q = 7 > z_val + 2
        ({}, [good], [[]], V, -2),                                                          # empty configuration
        ({}, [good], [cfg], bad_v, -2),                                                     # V_ion not finite
        ({}, [_CPseudoAtom((0, 2, -1, -1), (2, 2, 0, 0), 4.0, 0.5, 0, 0)], [cfg], V, -2),  # row out of range
        ({}, [_CPseudoAtom((0, 1, -1, -1), (2, 1, 0, 0), 4.0, 0.5, 0, 0)], [cfg], V, -2),  # n_ref below l + 1
        ({}, [_CPseudoAtom((-1, -1, -1, -1), (0, 0, 0, 0), 4.0, 0.5, 0, 0)], [cfg], V, -2),  # no channel
        ({}, [_CPseudoAtom((0, 1, -1, -1), (2, 2, 0, 0), 4.0, 0.5, 2, 0)], [cfg], V, -2),  # method 2
        ({}, [_CPseudoAtom((0, 1, -1, -1), (2, 2, 0, 0), 0.0, 0.5, 0, 0)], [cfg], V, -2),  # z_val 0
        ({}, [good], [cfg], deep, -2),                                                      # Z_b > 118
        ({}, [good, good], [cfg, [(2, 0, 0, 2.0), (2, 1, 0, 9.0)]], V, -2),                # the second atom is bad
    ]
    for kw, atoms, cfgs, v, want in cases:
        rc, untouched = _raw(ctx, v, atoms, cfgs, **kw)
        assert rc == want and untouched, (kw, rc, D.api.load_library().dftatom_last_error())
    small = _CRadial()
    small.orbitals = np.zeros(16385).ctypes.data_as(C.POINTER(C.c_double)); small.orbital_rows = 1
    rc, untouched = _raw(ctx, V, [good], [cfg], radial=C.byref(small))
    assert rc == -5 and untouched


def test_cli_table_equals_the_python_calls(ctx):
    exe = os.path.join(ROOT, "bin", "dftatom")
    o, _, pp = _pp(ctx, "Si")
    tests = ["3s1 3p3 3d0", "3s2 3p1 3d0"]
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([exe, "--Z", "14", "--levels", "14", "--delta", "0.0005", "--rmax", "25", "--config", "[Ne] 3s2 3p2 3d0", "--quiet-steps",
                        "--pseudo", tmp, "--pseudo-rc", "2.2", "--pseudo-test", ";".join(tests)], check=True, capture_output=True)
        lines = open(os.path.join(tmp, "0_Z14_pseudo_test.tsv")).read().splitlines()
    rows = [ln.split("\t") for ln in lines if not ln.startswith("#")]
    levels = [ln.split("\t")[1:] for ln in lines if ln.startswith("# level\t") and not ln.startswith("# level\tconfig")]
    valence = [_ref_valence(pp) + "", *tests]
    ps = ctx.solve_pseudo_batch(pp, valence)
    ae = _solve_ae(ctx, "Si", valence)
    assert [r[0] for r in rows[1:]] == tests
    for q, row in enumerate(rows):
        assert float(row[2]) == ae[q].Etotal and float(row[3]) == ps[q].Etotal, (q, row)
        assert float(row[4]) == ae[q].Etotal - ae[0].Etotal and float(row[5]) == ps[q].Etotal - ps[0].Etotal
        assert int(row[7]) == ae[q].status and int(row[8]) == ps[q].status
    want = []
    for q, (rp, ra) in enumerate(zip(ps, ae)):
        for L in rp.levels[0]:
            e_ae = [x.E for x in ra.levels[0] if (x.n, x.l) == (L.n, L.l)][0]
            want.append((L.n, L.l, L.E, e_ae))
    got = [(int(x[1]), int(x[2]), float(x[6]), float(x[5])) for x in levels]
    assert got == want
