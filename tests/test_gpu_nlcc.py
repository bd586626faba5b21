"""GPU tests of the nonlinear core correction (Context.partial_core / dftatom_partial_core, Context.pseudize(..., r_pc) /
dftatom_tm_pseudize_core, Context.solve_pseudo_batch with a core / dftatom_solve_pseudo_batch_core): the partial core against the numpy
reference of tests/nlcc_ref.py, the calls without a core against the calls of the parent entries (bit for bit), the reference
configuration and parity of the core-corrected pseudo-atom, the transferability of Na and Cu with no core, the partial core and the full
core, the CLI flag --pseudo-core, and the argument validation of the three entry points."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import logderiv_ref as LR
import nlcc_ref as NR
from dftatom_b200.api import _CConfig, _CCoreOrbital, _COccupation, _CPccResult, _CPseudoAtom, _CResult, _CStep, _CTmChannel, _CTmResult

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRID = (14, 0.0005, 25.0)
ATOMS = {
    "C": (D.Options(6, *GRID[:1], GRID[2], GRID[1], 0.5, 0), 1.8),
    "Si": (D.Options(14, GRID[0], GRID[2], GRID[1], 0.5, 0, config="[Ne] 3s2 3p2 3d0"), 2.2),
    "Na": (D.Options(11, GRID[0], GRID[2], GRID[1], 0.5, 0, config="[Ne] 3s1 3p0"), 2.8),
    "Cu": (D.Options(29, GRID[0], GRID[2], GRID[1], 0.5, 0, config="[Ar] 3d10 4s1 4p0"), 2.2),
}
CORE = {"C": "[He]", "Si": "[Ne]", "Na": "[Ne]", "Cu": "[Ar]"}
ADAPTIVE = {"Cu"}
EPS_TOL = 7.5e-6          # tests/test_gpu_pseudo_scf.py

_ae, _pp = {}, {}


def _adaptive(ctx, name):
    ctx.set_option("adaptive_mixing", int(name in ADAPTIVE))


def _solve_ae_ref(ctx, name):
    if name not in _ae:
        _adaptive(ctx, name)
        try:
            res = ctx.solve_batch([ATOMS[name][0]], keep_steps=False, radial=True)[0]
        finally:
            ctx.set_option("adaptive_mixing", 0)
        assert res.finished
        _ae[name] = res
    return _ae[name]


def r_pc_rule(ctx, name):
    """The partial-core radius of these tests: the outermost node where rho_core >= rho_val (the valence density of the pseudization
    without a core)."""
    pp = pseudo(ctx, name, None)
    rc = pp_core(ctx, name).rho_core[0]
    rv = pp.rho_val[0]
    i = max(k for k in range(1, len(rc) - 1) if rc[k] >= rv[k])
    return float(pp.r[i])


def pp_core(ctx, name):
    return pseudo(ctx, name, 0.0).core


def pseudo(ctx, name, r_pc):
    """Pseudopotential of `name`: r_pc None = no core, 0 = the full core, "lfc" = the partial core at r_pc_rule."""
    key = (name, r_pc)
    if key not in _pp:
        rr = r_pc_rule(ctx, name) if r_pc == "lfc" else r_pc
        pp = ctx.pseudize(_solve_ae_ref(ctx, name), ATOMS[name][1], r_pc=rr)
        assert np.all(pp.status == 0)
        _pp[key] = pp
    return _pp[key]


def _ref_valence(pp):
    return " ".join(f"{n}{'spdf'[l]}{occ:g}" for n, l, occ in sorted(zip(pp.n.tolist(), pp.l.tolist(), pp.occ.tolist())))


def _solve(ctx, name, fn):
    _adaptive(ctx, name)
    try:
        return fn()
    finally:
        ctx.set_option("adaptive_mixing", 0)


@pytest.fixture(scope="module")
def ctx():
    with D.Context(0) as c:
        yield c


def test_partial_core_matches_the_reference(ctx):
    levels, delta, max_r = GRID
    out = []
    for name in ("Na", "Si", "Cu"):
        res = _solve_ae_ref(ctx, name)
        pp = pseudo(ctx, name, None)
        valence = {int(n) * 10 + int(l) for n, l in zip(pp.n, pp.l)}
        core = [k for k, L in enumerate(res.levels[0]) if L.n * 10 + L.l not in valence]
        occ = [float(res.levels[0][k].occ) for k in core]
        u = res.radial.orbitals[0]
        rule = r_pc_rule(ctx, name)
        pc = ctx.partial_core(u, levels, delta, max_r, [0] * len(core) + [1] * len(core), core * 2, occ * 2, [0.0, rule])
        rho_core = NR.core_density([u[k] for k in core], occ, levels, delta, max_r)
        np.testing.assert_allclose(pc.rho_core[0], rho_core, rtol=1e-12, atol=0)
        for p, r_pc in enumerate((0.0, rule)):
            ref = NR.partial_core(rho_core, levels, delta, max_r, r_pc)
            assert pc.status[p] == ref["status"] == 0 and pc.i_pc[p] == ref["i_pc"]
            assert pc.r_pc[p] == ref["r_pc"]
            if r_pc > 0:
                assert abs(pc.A[p] - ref["A"]) <= 1e-12 * abs(ref["A"]) and abs(pc.B[p] - ref["B"]) <= 1e-12 * abs(ref["B"])
            np.testing.assert_allclose(pc.rho_pc[p], ref["rho_pc"], rtol=1e-12, atol=0)
            assert abs(pc.n_core[p] - ref["n_core"]) <= 1e-12 * ref["n_core"]
            assert abs(pc.n_pc[p] - ref["n_pc"]) <= 1e-12 * ref["n_pc"]
        want = sum(occ)
        out.append((name, want, pc.n_core[0], rule, pc.n_pc[1]))
    print("MEASURED n_core: " + "; ".join(f"{n} {w:g} electrons: n_core - Q {c - w:+.2e}, r_pc {r:.4f}, n_pc {p:.6f}" for n, w, c, r, p in out))
    # measured on a B200 at 1000 W: n_core - Q = -1.8e-15 (Na), 0 (Si), 0 (Cu); stated tolerance 1e-13 electrons
    for n, w, c, _, _ in out:
        assert abs(c - w) < 1e-13, (n, w, c)
    # a density that rises at r_pc: status 1, NaN row, A and B
    N = len(pp.r)
    bad = ctx.partial_core(np.array([pp.r ** 3]), levels, delta, max_r, 0, 0, 1.0, [1.0])
    assert bad.status[0] == 1 and np.isnan(bad.A[0]) and np.isnan(bad.B[0]) and np.all(np.isnan(bad.rho_pc[0][1:N]))


def _raw_tm(ctx, V, u, ch, rho_pc, core):
    levels, delta, max_r = GRID
    nc, N = len(ch), V.shape[1]
    res = np.zeros(nc, dtype=np.dtype(_CTmResult))
    rows = [np.zeros((nc, N)) for _ in range(3)] + [np.zeros(V.shape)]
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    args = [ctx._h, levels, delta, max_r, dp(V), V.shape[0], dp(u), u.shape[0], ch.ctypes.data_as(C.POINTER(_CTmChannel)), nc,
            res.ctypes.data_as(C.POINTER(_CTmResult))] + [dp(x) for x in rows]
    rc = ctx._lib.dftatom_tm_pseudize_core(*args, rho_pc) if core else ctx._lib.dftatom_tm_pseudize(*args)
    assert rc == 0
    return res.tobytes(), [x.tobytes() for x in rows]


def _raw_ps(ctx, pps, cfgs, rho_pc=None, pc_row=None, core=False):
    levels, delta, max_r = GRID
    n = len(pps)
    rows, ca = [], (_CPseudoAtom * n)()
    for a, pp in enumerate(pps):
        ca[a].row[:] = [-1] * 4
        for c, l in enumerate(pp.l.tolist()):
            ca[a].row[l] = len(rows) + c
            ca[a].n_ref[l] = int(pp.n[c])
        rows += list(pp.V_ion)
        ca[a].z_val = float(np.sum(pp.occ)); ca[a].mixing = 0.5; ca[a].method = 0
    cc = (_CConfig * n)()
    for a, cfg in enumerate(cfgs):
        e = [(x[0], x[1], 0, x[2]) for x in D.parse_config(cfg)]
        cc[a].n_orbitals = len(e)
        for k, x in enumerate(e):
            cc[a].orb[k] = _COccupation(*x)
    V = np.ascontiguousarray(rows)
    out = (_CResult * n)()
    steps = (_CStep * (n * 100))()
    from dftatom_b200.api import _radial_buffers
    views, crad = _radial_buffers(n, V.shape[1], sum(cc[a].n_orbitals for a in range(n)))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    args = [ctx._h, levels, delta, max_r, dp(V), V.shape[0], ca, cc, n, out, steps, 100, C.byref(crad)]
    if core:
        PC = None if rho_pc is None else np.ascontiguousarray(rho_pc)
        PR = None if pc_row is None else np.ascontiguousarray(pc_row, np.int32)
        rc = ctx._lib.dftatom_solve_pseudo_batch_core(*args, None if PC is None else dp(PC), 0 if PC is None else PC.shape[0],
                                                      None if PR is None else PR.ctypes.data_as(C.POINTER(C.c_int)))
    else:
        rc = ctx._lib.dftatom_solve_pseudo_batch(*args)
    assert rc == 0, D.api.load_library().dftatom_last_error()
    return bytes(out), bytes(steps), [np.array(v) for v in views]


def test_no_core_changes_nothing(ctx):
    res = _solve_ae_ref(ctx, "Si")
    pp = pseudo(ctx, "Si", None)
    ch = np.zeros(len(pp.l), dtype=np.dtype(_CTmChannel))
    best = [k for k, L in enumerate(res.levels[0]) for c in range(len(pp.l)) if (L.n, L.l) == (pp.n[c], pp.l[c])]
    ch["pot"], ch["orbital"], ch["l"], ch["eps"], ch["occ"], ch["r_c"] = 0, best, pp.l, pp.eps, pp.occ, ATOMS["Si"][1]
    V, u = np.ascontiguousarray([res.radial.V[0]]), np.ascontiguousarray(res.radial.orbitals[0])
    assert _raw_tm(ctx, V, u, ch, None, False) == _raw_tm(ctx, V, u, ch, None, True)
    cfgs = ["3s2 3p2 3d0", "3s1 3p3 3d0"]
    old = _raw_ps(ctx, [pp, pp], cfgs)
    pcr = pseudo(ctx, "Si", 0.0).rho_pc
    for kw in (dict(), dict(rho_pc=pcr, pc_row=[-1, -1])):
        new = _raw_ps(ctx, [pp, pp], cfgs, core=True, **kw)
        assert new[0] == old[0] and new[1] == old[1]
        assert all(np.array_equal(a, b) for a, b in zip(old[2], new[2]))
    # an atom without a core inside a batch with cores equals that atom alone
    ppc = pseudo(ctx, "Si", "lfc")
    for method, cfg, cfg_c in ((0, "3s1 3p3 3d0", "3s2 3p2 3d0"), (1, "3s1/0 3p2/1 3d0/0", "3s1/1 3p2/0 3d0/0")):
        alone = ctx.solve_pseudo_batch(pp, cfg, method=method, radial=True)[0]
        mixed = ctx.solve_pseudo_batch([ppc, pp, ppc], [cfg_c, cfg, cfg], method=method, radial=True)
        b = mixed[1]
        assert alone.n_steps == b.n_steps and alone.status == b.status
        for k in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"):
            assert getattr(alone, k) == getattr(b, k), (method, k)
        assert len(alone.steps) == len(b.steps)
        for x, y in zip(alone.steps, b.steps):
            assert x == y, method
        assert [L.E for s in alone.levels for L in s] == [L.E for s in b.levels for L in s]
        ra, rb = alone.radial, b.radial
        for f in ("rho", "V", "V_H"):
            assert np.array_equal(getattr(ra, f), getattr(rb, f)), (method, f)
        for f in ("orbitals", "moments"):
            assert all(np.array_equal(x, y) for x, y in zip(getattr(ra, f), getattr(rb, f))), (method, f)
        assert (ra.n_electrons, ra.r2) == (rb.n_electrons, rb.r2)
        assert mixed[2].Etotal != b.Etotal


def test_core_corrected_unscreening_matches_the_reference(ctx):
    """V_ion of dftatom_tm_pseudize_core against nlcc_ref.unscreen_core on two potential rows of Si: row 0 without electrons (every
    occupation 0: V_H = 0) and the full core, row 1 the reference valence with the partial core, so the rows' Poisson slots are swapped."""
    levels, delta, max_r = GRID
    res = _solve_ae_ref(ctx, "Si")
    pp = pseudo(ctx, "Si", None)
    best = [k for c in range(len(pp.l)) for k, L in enumerate(res.levels[0]) if (L.n, L.l) == (pp.n[c], pp.l[c])]
    nc = len(pp.l)
    V = np.array([res.radial.V[0], res.radial.V[0]])
    pc = np.array([pseudo(ctx, "Si", 0.0).rho_pc[0], pseudo(ctx, "Si", "lfc").rho_pc[0]])
    occ = np.concatenate([np.zeros(nc), pp.occ])
    out = ctx.tm_pseudize(V, res.radial.orbitals[0], *GRID, [0] * nc + [1] * nc, best * 2, np.tile(pp.l, 2), np.tile(pp.eps, 2), occ,
                          ATOMS["Si"][1], rho_pc=pc)
    assert np.all(out.status == 0)
    r = out.r
    worst = 0.0
    for p in range(2):
        chans = [(dict(status=0, u_ps=out.u[c], v_scr=out.V_scr[c]), int(out.l[c]), float(occ[c])) for c in range(p * nc, (p + 1) * nc)]
        rho, vh, vxc, vion = NR.unscreen_core(levels, delta, max_r, chans, pc[p])
        assert np.all(np.abs(out.rho_val[p] - rho) <= 1e-12 * max(rho.max(), 1e-300))
        Qv = float(sum(x[2] for x in chans))
        # the floor of the cold multigrid solve against the exact discrete solution, as tests/test_gpu_pseudo.py states it
        tol = 2e-9 * max(1.0, Qv) / np.where(r > 0, r, 1.0)
        for k in range(nc):
            tol_k = tol + 1e-9 * np.maximum(1.0, np.abs(vion[k]))
            d = np.abs(out.V_ion[p * nc + k][1:] - vion[k][1:])
            assert np.all(d <= tol_k[1:]), (p, k, d.max())
            worst = max(worst, float(np.max(d / tol_k[1:])))
    print(f"MEASURED core-corrected V_ion against the reference: at most {worst:.2f} of the Poisson-floor tolerance")
    assert not np.any(out.rho_val[0])


# measured on a B200 at 1000 W, max over the channels |eps_PS - eps_AE|: with the partial core at the r_pc rule C 7.1e-10, Cu 3.0e-8,
# Na 5.1e-11, Si 2.1e-6 (the empty 3d box state, as without a core) - within EPS_TOL; with the full core C 7.3e-10, Cu 2.9e-8, Na 2.9e-10
# and Si 1.8e-5, above EPS_TOL (bound 5.4e-5, 3x the measured value).  The cause is the stop test: it is relative, |dE/E| < 1e-11, and
# the full core's xc energy makes Si's Etotal -22.05 Ha (without a core the pseudo-atom's is -3.5 Ha in 3s1 3p3), so the SCF stops at a
# several times larger absolute energy change, and the unbound 3d box state, which follows the density tail, is the level still moving.  Run to the 100-step cap the same full-core
# pseudo-atom is within 3.0e-6 Ha (C 7.0e-10, Cu 3.1e-8, Na 5.3e-11), inside EPS_TOL, which the test asserts.
FULL_CORE_EPS_TOL = 5.4e-5


@pytest.mark.parametrize("name", sorted(ATOMS))
def test_reference_configuration_with_a_core_reproduces_the_all_electron_atom(ctx, name):
    errs = []
    for kind in ("lfc", 0.0):
        pp = pseudo(ctx, name, kind)
        r = _solve(ctx, name, lambda: ctx.solve_pseudo_batch(pp, _ref_valence(pp), radial=True)[0])
        assert r.finished, r.status
        lev = {(L.n, L.l): L for L in r.levels[0]}
        errs.append(max(abs(lev[(n, l)].E - pp.eps[c]) for c, (l, n) in enumerate(zip(pp.l.tolist(), pp.n.tolist()))))
        assert abs(r.Ekin + r.Eenuc + r.Ecoul + r.Exc - r.Etotal) < 1e-8
    # the same full-core pseudo-atom run to the step cap: the relative stop test |dE/E| < 1e-11 stops later in absolute terms when
    # the core's xc energy makes |Etotal| large
    pp = pseudo(ctx, name, 0.0)
    ctx.set_option("run_to_cap", 1)
    try:
        r = _solve(ctx, name, lambda: ctx.solve_pseudo_batch(pp, _ref_valence(pp))[0])
    finally:
        ctx.set_option("run_to_cap", 0)
    lev = {(L.n, L.l): L for L in r.levels[0]}
    cap = max(abs(lev[(n, l)].E - pp.eps[c]) for c, (l, n) in enumerate(zip(pp.l.tolist(), pp.n.tolist())))
    print(f"MEASURED reference with core {name}: LFC r_pc {pseudo(ctx, name, 'lfc').core.r_pc[0]:.4f} eps {errs[0]:.3e}, full core eps "
          f"{errs[1]:.3e} (Etotal {r.Etotal:.6f}; run to the cap, {r.n_steps} steps: eps {cap:.3e})")
    assert errs[0] <= EPS_TOL
    assert errs[1] <= FULL_CORE_EPS_TOL
    assert cap <= EPS_TOL


# measured on a B200 at 1000 W (max over the cases): eigenvalues 1.5e-9 Ha, energies 4.6e-9 Ha, Etotal = Ekin + Eenuc + Ecoul + Exc to 3e-11
@pytest.mark.parametrize("name,config,method", [("C", "2s2 2p2", 0), ("Si", "3s1 3p3", 0), ("C", "2s1/1 2p2/0", 1), ("Si", "3s1/1 3p2/0", 1)])
def test_parity_with_the_numpy_reference(ctx, name, config, method):
    o = ATOMS[name][0]
    pp = pseudo(ctx, name, "lfc")
    r = ctx.solve_pseudo_batch(pp, config, method=method)[0]
    assert r.finished
    v_ion = {int(l): pp.V_ion[c] for c, l in enumerate(pp.l.tolist())}
    n_ref = {int(l): int(n) for l, n in zip(pp.l.tolist(), pp.n.tolist())}
    entries = [e if len(e) == 4 else (e[0], e[1], 0, e[2]) for e in D.parse_config(config, method)]
    ref = NR.solve(v_ion, n_ref, entries, o.MultigridLevels, o.deltaGrid, o.MaxR, pp.rho_pc[0], mixing=0.5, method=method)
    assert ref["converged"]
    de = max(abs(L.E - ref["E"][s][k]) for s, ch in enumerate(r.levels) for k, L in enumerate(ch))
    dE = max(abs(getattr(r, k) - ref[k]) for k in ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc"))
    ident = abs(r.Ekin + r.Eenuc + r.Ecoul + r.Exc - r.Etotal)
    print(f"MEASURED parity with core {name} {config} method {method}: eps {de:.3e} energies {dE:.3e} identity {ident:.1e}")
    assert de < 1e-6 and dE < 1e-5 and ident < 1e-8


# (name, method, reference valence, test valence): spin polarisation and excitation energies against the all-electron atom
CASES = [
    ("Na", 1, "3s0.5/0.5 3p0/0", "3s1/0 3p0/0"),
    ("Na", 0, "3s1 3p0", "3s0 3p1"),
    ("Cu", 0, "3d10 4s1 4p0", "3d9 4s2 4p0"),
    ("Cu", 1, "3d5/5 4s0.5/0.5 4p0/0", "3d5/5 4s1/0 4p0/0"),
]


# measured on a B200 at 1000 W, |dE_PS - dE_AE| in Ha for no core / LFC at the r_pc rule / full core:
#   Na spin polarisation (LSDA 3s1/0 against 3s0.5/0.5)  1.34e-3 / 1.09e-4 / 3.31e-5
#   Na 3s -> 3p                                           1.90e-3 / 5.79e-5 / 1.98e-4
#   Cu 3d9 4s2 (against 3d10 4s1)                         1.41e-3 / 2.18e-3 / 2.19e-3
#   Cu 4s spin polarisation (LSDA, 3d5/5)                 1.38e-5 / 1.34e-4 / 1.34e-4
# Na follows the literature: the core correction removes most of the spin-polarisation error.  Cu's 4s spin polarisation contradicts
# it (a finding): with 3d in the valence the no-core error is already 1.4e-5 Ha, and the core correction adds 1.2e-4 Ha; the ordering is
# asserted for Na, and kept for Cu as a strict expected failure.  Bounds: 3x the measured values.
BOUNDS = {("Na", 1): (4e-3, 3.3e-4, 1e-4), ("Na", 0): (5.7e-3, 1.8e-4, 6e-4), ("Cu", 0): (4.2e-3, 6.6e-3, 6.6e-3), ("Cu", 1): (4.2e-5, 4e-4, 4e-4)}


def test_transferability_with_and_without_the_core(ctx):
    rows = []
    for name, method, ref, cfg in CASES:
        o = ATOMS[name][0]
        opts = [D.Options(o.Z, o.MultigridLevels, o.MaxR, o.deltaGrid, o.alpha, method, config=f"{CORE[name]} {v}") for v in (ref, cfg)]
        ae = _solve(ctx, name, lambda: ctx.solve_batch(opts, keep_steps=False))
        assert all(x.finished for x in ae), [(x.status, x.n_steps) for x in ae]
        d_ae = ae[1].Etotal - ae[0].Etotal
        err = []
        for kind in (None, "lfc", 0.0):
            ps = _solve(ctx, name, lambda: ctx.solve_pseudo_batch(pseudo(ctx, name, kind), [ref, cfg], method=method))
            assert all(x.finished for x in ps), [(x.status, x.n_steps) for x in ps]
            err.append(abs((ps[1].Etotal - ps[0].Etotal) - d_ae))
        rows.append((name, method, cfg, d_ae, err))
    print("MEASURED transferability |dE_PS - dE_AE| (Ha): no core / LFC / full core: "
          + "; ".join(f"{n} m{m} {c}: dE_AE {d:.6f} {e[0]:.2e} / {e[1]:.2e} / {e[2]:.2e}" for n, m, c, d, e in rows))
    for n, m, c, d, e in rows:
        assert all(x <= b for x, b in zip(e, BOUNDS[(n, m)])), (n, c, e)
    _transfer.update({(n, m): e for n, m, c, d, e in rows})
    e = _transfer[("Na", 1)]            # spin polarisation of an alkali atom: the literature's case for the core correction
    assert e[1] < e[0] and e[2] < e[0], e


_transfer = {}


@pytest.mark.xfail(strict=True, reason="measured: Cu's 4s spin-polarisation error grows with the core (1.4e-5 Ha without, 1.3e-4 Ha "
                                       "with the partial or the full core); with 3d in the valence the core adds little xc nonlinearity")
def test_the_core_reduces_the_cu_4s_spin_polarisation_error(ctx):
    if ("Cu", 1) not in _transfer:
        test_transferability_with_and_without_the_core(ctx)
    e = _transfer[("Cu", 1)]
    assert e[1] < e[0] and e[2] < e[0], e


def test_cli_core_table_equals_the_python_calls(ctx):
    exe = os.path.join(ROOT, "bin", "dftatom")
    tests = ["3s0 3p1"]
    rule = r_pc_rule(ctx, "Na")
    args = [exe, "--Z", "11", "--levels", "14", "--delta", "0.0005", "--rmax", "25", "--config", "[Ne] 3s1 3p0", "--quiet-steps",
            "--pseudo-rc", "2.8", "--pseudo-test", ";".join(tests)]
    with tempfile.TemporaryDirectory() as tmp:
        a, b = os.path.join(tmp, "a"), os.path.join(tmp, "b")
        os.mkdir(a); os.mkdir(b)
        subprocess.run(args + ["--pseudo", a], check=True, capture_output=True)
        subprocess.run(args + ["--pseudo", b, "--pseudo-core", repr(rule)], check=True, capture_output=True)
        plain = open(os.path.join(a, "0_Z11_pseudo.tsv")).read().splitlines()
        cored = open(os.path.join(b, "0_Z11_pseudo.tsv")).read().splitlines()
        lines = open(os.path.join(b, "0_Z11_pseudo_test.tsv")).read().splitlines()
    assert not any(x.startswith("# core") for x in plain)
    head = [x for x in plain if x.startswith("# r")][0].split("\t")
    assert head[-1] == "rho_val"
    core_line = [x.split("\t") for x in cored if x.startswith("# core")]
    pp = pseudo(ctx, "Na", "lfc")
    assert len(core_line) == 1 and float(core_line[0][1]) == pp.core.r_pc[0] and float(core_line[0][3]) == pp.core.A[0]
    data = np.array([[float(v) for v in x.split("\t")] for x in cored if not x.startswith("#")])
    assert np.array_equal(data[:, -2], pp.rho_core[0]) and np.array_equal(data[:, -1], pp.rho_pc[0])
    rows = [ln.split("\t") for ln in lines if not ln.startswith("#")]
    ps = ctx.solve_pseudo_batch(pp, [_ref_valence(pp), *tests])
    for q, row in enumerate(rows):
        assert float(row[3]) == ps[q].Etotal, (q, row)


def test_invalid_arguments_are_rejected_before_any_launch(ctx):
    """Every rule of the validation of dftatom_partial_core, the rho_pc rows of dftatom_tm_pseudize_core and pc_row / rho_pc of
    dftatom_solve_pseudo_batch_core: the return code, the row, entry or atom (and node) the message names, and the outputs untouched."""
    lib = D.load_library()
    dp = C.POINTER(C.c_double)
    levels, delta, max_r = 12, 0.002, 25.0
    N, r, _, _ = LR.grid(levels, delta, max_r)
    u = np.stack([r * r * np.exp(-r / 2), r * (1 - r / 2) * np.exp(-r / 2)])

    def pc_call(u=u, n_orb=2, core=((0, 0, 2.0), (1, 1, 1.0)), n_core=None, r_pc=(0.0, 1.5), n_rows=None, null=()):
        u = np.ascontiguousarray(u, dtype=np.float64)
        cc = np.zeros(max(1, len(core)), dtype=np.dtype(_CCoreOrbital))
        for k, e in enumerate(core):
            cc[k] = e
        rp = np.ascontiguousarray(r_pc, dtype=np.float64)
        n_core = len(core) if n_core is None else n_core
        n_rows = len(r_pc) if n_rows is None else n_rows
        out = np.full(max(1, len(r_pc)), 7.0, dtype=np.dtype(_CPccResult))
        rows = [np.full((max(1, len(r_pc)), N), 7.0) for _ in range(2)]
        args = {"u": u.ctypes.data_as(dp), "core": cc.ctypes.data_as(C.POINTER(_CCoreOrbital)), "r_pc": rp.ctypes.data_as(dp),
                "out": out.ctypes.data_as(C.POINTER(_CPccResult))}
        for k in null:
            args[k] = None
        rc = lib.dftatom_partial_core(ctx._h, levels, delta, max_r, args["u"], n_orb, args["core"], n_core, args["r_pc"], n_rows, args["out"],
                                      *[x.ctypes.data_as(dp) for x in rows])
        untouched = bool(np.all(out["A"] == 7.0) and all(np.all(x == 7.0) for x in rows))
        return rc, lib.dftatom_last_error().decode(), untouched

    rc, msg, _ = pc_call()
    assert rc == 0, msg
    bad_u = u.copy(); bad_u[1, 9] = np.inf
    cases = [
        (dict(null=("u",)), "NULL"),
        (dict(null=("r_pc",)), "NULL"),
        (dict(null=("out",)), "NULL"),
        (dict(null=("core",)), "NULL"),                                         # core = NULL with n_core > 0
        (dict(n_orb=0), "n_orb"),
        (dict(n_rows=0), "n_rows"),
        (dict(n_core=-1), "n_core"),
        (dict(r_pc=(0.0, np.nan)), "row 1: r_pc"),
        (dict(r_pc=(-0.5, 1.5)), "row 0: r_pc"),
        (dict(r_pc=(0.0, 0.5 * (r[2] + r[3]))), "row 1: r_pc"),                 # inside (0, r_3)
        (dict(r_pc=(0.0, r[N - 3] * 1.0001)), "row 1: r_pc"),                   # above r_(N-3)
        (dict(core=((0, 0, 2.0), (2, 1, 1.0))), "core entry 1: row"),
        (dict(core=((-1, 0, 2.0), (1, 1, 1.0))), "core entry 0: row"),
        (dict(core=((0, 0, 2.0), (1, 2, 1.0))), "core entry 1: orbital"),
        (dict(core=((0, -1, 2.0), (1, 1, 1.0))), "core entry 0: orbital"),
        (dict(core=((0, 0, -0.5), (1, 1, 1.0))), "core entry 0: occ"),
        (dict(core=((0, 0, 2.0), (1, 1, 14.5))), "core entry 1: occ"),
        (dict(core=((0, 0, np.nan), (1, 1, 1.0))), "core entry 0: occ"),
        (dict(u=bad_u), "orbital row 1: u is not finite at node 9"),
    ]
    for kw, text in cases:
        rc, msg, untouched = pc_call(**kw)
        assert rc == -5, (kw, rc, msg)
        assert text in msg, (kw, msg)
        assert untouched, kw

    # dftatom_tm_pseudize_core: a rho_pc row not finite or negative at a node >= 1
    V = np.zeros((2, N))
    V[:, 1:] = -1.0 / r[1:]
    ch = np.zeros(1, dtype=np.dtype(_CTmChannel))
    ch[0] = (0, 0, 1, 0, -0.125, 1.0, 2.0)

    def tm_call(rho_pc):
        rho_pc = np.ascontiguousarray(rho_pc, dtype=np.float64)
        out = np.full(1, 7.0, dtype=np.dtype(_CTmResult))
        rows = [np.full((1, N), 7.0) for _ in range(3)] + [np.full((2, N), 7.0)]
        rc = lib.dftatom_tm_pseudize_core(ctx._h, levels, delta, max_r, V.ctypes.data_as(dp), 2, u.ctypes.data_as(dp), 2,
                                          ch.ctypes.data_as(C.POINTER(_CTmChannel)), 1, out.ctypes.data_as(C.POINTER(_CTmResult)),
                                          *[x.ctypes.data_as(dp) for x in rows], rho_pc.ctypes.data_as(dp))
        untouched = bool(np.all(out["q"] == 7.0) and all(np.all(x == 7.0) for x in rows))
        return rc, lib.dftatom_last_error().decode(), untouched

    pc = np.zeros((2, N))
    rc, msg, _ = tm_call(pc)
    assert rc == 0, msg
    for row, node, x in ((1, 9, np.nan), (0, 3, -1e-30), (1, N - 1, np.inf)):
        bad = pc.copy(); bad[row, node] = x
        rc, msg, untouched = tm_call(bad)
        assert rc == -5 and untouched, (row, node, rc, msg)
        assert f"rho_pc row {row}: " in msg and f"at node {node}" in msg, msg

    # dftatom_solve_pseudo_batch_core: pc_row out of range, a rho_pc row not finite or negative
    pp = pseudo(ctx, "Si", None)
    pcr = pseudo(ctx, "Si", 0.0).rho_pc
    n = 2
    ca = (_CPseudoAtom * n)()
    for a in range(n):
        ca[a].row[:] = [-1] * 4
        for c_, l in enumerate(pp.l.tolist()):
            ca[a].row[l] = c_
            ca[a].n_ref[l] = int(pp.n[c_])
        ca[a].z_val = float(np.sum(pp.occ)); ca[a].mixing = 0.5; ca[a].method = 0
    cc = (_CConfig * n)()
    for a in range(n):
        e = [(x[0], x[1], 0, x[2]) for x in D.parse_config("3s2 3p2 3d0")]
        cc[a].n_orbitals = len(e)
        for k, x in enumerate(e):
            cc[a].orb[k] = _COccupation(*x)
    VI = np.ascontiguousarray(pp.V_ion)

    def ps_call(rho_pc, pc_row):
        out = (_CResult * n)()
        C.memset(out, 0x5A, C.sizeof(out))
        PC = None if rho_pc is None else np.ascontiguousarray(rho_pc, dtype=np.float64)
        PR = np.ascontiguousarray(pc_row, np.int32)
        rc = lib.dftatom_solve_pseudo_batch_core(ctx._h, *GRID, VI.ctypes.data_as(dp), VI.shape[0], ca, cc, n, out, None, 0, None,
                                                 None if PC is None else PC.ctypes.data_as(dp), 0 if PC is None else PC.shape[0],
                                                 PR.ctypes.data_as(C.POINTER(C.c_int)))
        return rc, lib.dftatom_last_error().decode(), all(b == 0x5A for b in bytes(out))

    two = np.stack([pcr[0], pcr[0]])
    assert ps_call(two, [0, 1])[0] == 0
    nan_row = two.copy(); nan_row[1, 50] = np.nan
    neg_row = two.copy(); neg_row[0, 4] = -1e-3
    cases = [
        ((two, [0, 2]), "atom 1: pc_row = 2"),
        ((two, [-2, 1]), "atom 0: pc_row = -2"),
        ((None, [0, -1]), "atom 0: pc_row = 0"),                                # no rho_pc: only -1 is in range
        ((nan_row, [0, -1]), "rho_pc row 1"),                                   # every row is checked, used or not
        ((neg_row, [-1, 1]), "rho_pc row 0"),
    ]
    for (rho_pc, pc_row), text in cases:
        rc, msg, untouched = ps_call(rho_pc, pc_row)
        assert rc == -2 and untouched, (pc_row, rc, msg)
        assert text in msg, (pc_row, msg)
    assert "at node 50" in ps_call(nan_row, [0, -1])[1] and "at node 4" in ps_call(neg_row, [-1, 1])[1]
