"""GPU tests of the Kleinman-Bylander form (Context.kb_form / Context.kleinman_bylander / Context.kb_log_derivatives): parity with the
numpy reference of tests/kb_ref.py on the converged, pseudized atoms of test_gpu_pseudo.py for every choice of the local channel, the
local channel against dftatom_log_derivatives, the reference energy against the semilocal channel, the GSS verdict against a dense
diagonalisation, a synthetic ghost, deep energies, independence of the batch, argument validation and the CLI tables."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dftatom_b200 as D
import kb_ref as K
import logderiv_ref as LR
from dftatom_b200.api import _CKbChannel, _CKbLdChannel, _CKbResult, _CLogDeriv

pytestmark = pytest.mark.gpu

ATOMS = {      # as tests/test_gpu_pseudo.py
    "C": (D.Options(6, 14, 25.0, 0.0005, 0.5, 0), 1.8),
    "Si": (D.Options(14, 14, 25.0, 0.0005, 0.5, 0, config="[Ne] 3s2 3p2 3d0"), 2.2),
    "Cu": (D.Options(29, 14, 25.0, 0.0005, 0.5, 0, config="[Ar] 3d10 4s1 4p0"), 2.2),
    "Ne-uniform": (D.Options(10, 14, 15.0, 0.0005, 0.5, 2), 1.8),
    "Rn": (D.Options(86, 17, 50.0, 0.0001, 0.5, 0), {0: 2.4, 1: 2.4, 2: 2.4, 3: 1.2}),
}
ADAPTIVE = {"Cu"}
GHOST_MARGIN = 1e-3        # Ha: the dense matrix's reference level sits within 1e-5 Ha of eps on these grids
_solved = {}


def _atom(ctx, name):
    if name not in _solved:
        o, r_c = ATOMS[name]
        ctx.set_option("adaptive_mixing", int(name in ADAPTIVE))
        try:
            res = ctx.solve_batch([o], keep_steps=False, radial=True)[0]
        finally:
            ctx.set_option("adaptive_mixing", 0)
        assert res.finished
        _solved[name] = (o, res, ctx.pseudize(res, r_c))
    return _solved[name]


def _zb(V):
    z = 1
    while -z * z - 1.0 > np.min(V[1:]):
        z += 1
    return z


@pytest.mark.parametrize("name", list(ATOMS))
def test_parity_local_channel_reference_state_and_ghosts(ctx, name):
    o, res, ps = _atom(ctx, name)
    grid = ps.grid
    # each channel 0.3 bohr beyond its own r_c: at E = eps the KB solution is a combination of the two outward chains that cancels their
    # growth in the classically forbidden region, so the rounding of that cancellation grows with the distance from the orbital's peak
    # (Rn 4f, r_c = 1.2 bohr: 3e-2 in D at 2.7 bohr between two correct sweeps, 1e-10 at 1.5 bohr)
    R = ps.r_c + 0.3
    for l_loc in ps.l.tolist():
        kb = ctx.kleinman_bylander(ps, l_loc)
        loc = int(np.nonzero(ps.l == l_loc)[0][0])
        E = np.concatenate([np.linspace(-2.0, 1.0, 7), ps.eps])
        ld = ctx.kb_log_derivatives(kb, ps.V_scr, R, E)
        sl = ctx.log_derivatives(ps.V_scr, *grid, np.arange(len(ps.l)), ps.l, R, E)
        for c, l in enumerate(ps.l.tolist()):
            ref = K.kb_form(ps.V_scr, ps.u, *grid, c, loc, l, ps.eps[c])
            # status 3 (the local search did not converge) is the engine's alone: the reference has no search
            assert kb.status[c] == ref["status"] or (ref["status"] == 0 and kb.status[c] == 3), (l_loc, c, kb.status[c])
            if c == loc:
                assert kb.E_KB[c] == 0 and kb.cos[c] == 1 and kb.ghost[c] == 0 and not kb.beta[c].any()
                # no projector: the sweep of dftatom_log_derivatives, bit for bit
                for f in ("D", "u", "du", "nodes"):
                    assert np.array_equal(getattr(ld, f)[c], getattr(sl, f)[c], equal_nan=True), (l_loc, f)
                continue
            assert ref["i_s"] == kb.i_s[c] and kb.r_s[c] == ps.r[ref["i_s"]]
            assert abs(kb.E_KB[c] - ref["E_KB"]) <= 1e-12 * abs(ref["E_KB"]) and abs(kb.cos[c] - ref["cos"]) <= 1e-12 * abs(ref["cos"])
            assert np.all(np.abs(kb.beta[c] - ref["beta"]) <= 1e-12 * np.abs(ref["beta"]).max())
            # the local eigenvalues: the SCF's search on the local row, as dftatom_level_search runs it
            Es, ok = ctx.level_search(ps.V_scr[loc], *grid, _zb(ps.V_scr[loc]), [l + 1, l + 2], [l, l])
            conv = bool(ok.all())
            assert kb.status[c] == (0 if conv else 3)
            assert np.all(np.abs(kb.eps_loc[c] - Es) <= 1e-10 * np.maximum(1.0, np.abs(Es))), (kb.eps_loc[c], Es)
            if conv:
                assert kb.ghost[c] == K.gss_ghost(kb.E_KB[c], ps.eps[c], kb.eps_loc[c])
                dense = K.dense_ghost(ps.V_scr[loc], kb.beta[c], *grid, l, kb.E_KB[c], ps.eps[c], GHOST_MARGIN, coarse_levels=11)
                assert kb.ghost[c] == dense, (name, l_loc, l, kb.E_KB[c], kb.eps_loc[c], ps.eps[c])
            # the KB log derivatives against the reference: 1e-9, widened where the combination is ill-conditioned.  Where
            # (sigma - E_KB h_p) u_h and E_KB h_h u_p, or sigma and E_KB h_p, cancel, the result carries the two sweeps' rounding times the
            # condition number `cond` of the combination; each sweep's own rounding grows at most linearly with its steps (n eps).  Measured:
            # <= 3.2e-10 everywhere except Rn 4f with s local at its eigenvalue (2.9e-7 in D at cond 7.7e5 after 1e5 steps)
            D_, u_, du_, n_, _, cond = K.kb_log_derivative(ps.V_scr[loc], kb.beta[c], *grid, l, kb.E_KB[c], R[c], E, return_cond=True)
            steps = max(LR.nearest_node(ps.r, R[c]), int(kb.i_s[c])) + 1
            tol = 1e-9 + cond * steps * np.finfo(float).eps
            for got, want in ((ld.D[c], D_), (ld.u[c], u_), (ld.du[c], du_)):
                err = np.abs(got - want) / np.maximum(1.0, np.abs(want))
                assert np.all(err <= tol), (l_loc, c, err.tolist(), cond.tolist())
            assert np.array_equal(ld.nodes[c], n_)
            # at E = eps_l the KB channel reproduces the semilocal V_scr,l at r_c, up to the difference the reference shows between the
            # two discretisations (the Numerov solution on V_scr,l at eps against the TM orbital the projector is built from), x 10
            k = len(E) - len(ps.eps) + c
            Dl, ul, dul, _, _ = LR.log_derivative(ps.V_scr[c], *grid, l, R[c], [E[k]])
            tol = [10 * abs(D_[k] - Dl[0]) + 1e-10 * abs(Dl[0]), 10 * abs(u_[k] - ul[0]) + 1e-10 * abs(ul[0]), 10 * abs(du_[k] - dul[0]) + 1e-10 * abs(dul[0])]
            assert abs(ld.D[c, k] - sl.D[c, k]) <= tol[0] and abs(ld.u[c, k] - sl.u[c, k]) <= tol[1] and abs(ld.du[c, k] - sl.du[c, k]) <= tol[2], (l_loc, c)


def test_synthetic_ghost_is_flagged(ctx):
    o, res, ps = _atom(ctx, "C")
    grid = ps.grid
    r = ps.r
    s, p = int(np.nonzero(ps.l == 0)[0][0]), int(np.nonzero(ps.l == 1)[0][0])
    eps = ps.eps[s]
    # the p potential as the local one, deepened by -A e^(-(r/0.5)^2) (exactly V_scr,p beyond ~3 bohr, where the Gaussian drops below
    # its rounding), with A the smallest of a ladder for which the reference puts the 1-node s level of the local potential below eps
    for A in (5.0, 10.0, 20.0, 40.0, 80.0):
        Vl = ps.V_scr[p] - A * np.exp(-(r / 0.5) ** 2)
        el = K.local_levels(Vl, *grid, 0)
        if el[1] < eps - 0.05:
            break
    V = np.stack([ps.V_scr[s], Vl])
    u = np.stack([ps.u[s], ps.u[s]])
    kb = ctx.kb_form(V, u, *grid, 0, 1, 0, eps)
    assert kb.status[0] == 0 and kb.E_KB[0] > 0
    assert np.all(np.abs(kb.eps_loc[0] - el) <= 1e-8 * np.abs(el))
    assert kb.ghost[0] == 1
    assert K.dense_ghost(Vl, kb.beta[0], *grid, 0, kb.E_KB[0], eps, GHOST_MARGIN, coarse_levels=11) == 1
    # below eps: the semilocal s channel has no level there, so its u(r_c) keeps its sign over [eps_0^loc - 1, eps); the KB channel has
    # the ghost level there, and the reference shows its solution at r_c passing through zero (a pole of D) in that window
    R = float(ps.r_c.max()) + 0.3
    E = np.linspace(el[0] - 1.0, eps - 1e-3, 201)
    ld = ctx.kb_log_derivatives(kb, V, R, E)
    sl = ctx.log_derivatives(ps.V_scr[s], *grid, 0, 0, R, E)
    assert np.all(np.sign(sl.u[0]) == np.sign(sl.u[0][0]))
    assert np.any(np.sign(ld.u[0][1:]) != np.sign(ld.u[0][:-1]))
    D_, u_, du_, n_, _ = K.kb_log_derivative(Vl, kb.beta[0], *grid, 0, kb.E_KB[0], R, E)
    assert np.all(np.abs(ld.D[0] - D_) <= 1e-9 * np.maximum(1.0, np.abs(D_))) and np.array_equal(ld.nodes[0], n_)


def test_deep_energies_stay_finite(ctx):
    o, res, ps = _atom(ctx, "Cu")
    grid = ps.grid
    kb = ctx.kleinman_bylander(ps, 0)
    loc = int(np.nonzero(ps.l == 0)[0][0])
    N = len(ps.r)
    R = ps.r[N - 2]                                          # the largest allowed r_c
    E = [-float(_zb(ps.V_scr[loc])) ** 2 - 1.0]
    ld = ctx.kb_log_derivatives(kb, ps.V_scr, R, E)
    for c in range(len(ps.l)):
        if c == loc:
            continue
        assert np.isfinite(ld.D[c, 0]) and np.isfinite(ld.u[c, 0]) and ld.nodes[c, 0] >= 0
        D_, u_, du_, n_, _ = K.kb_log_derivative(ps.V_scr[loc], kb.beta[c], *grid, int(ps.l[c]), kb.E_KB[c], R, E)
        assert abs(ld.D[c, 0] - D_[0]) <= 1e-9 * max(1.0, abs(D_[0])) and ld.nodes[c, 0] == n_[0]


def test_channel_is_independent_of_the_batch(ctx):
    # C3's valence channels pseudized as in scripts/gpu_kb_cost.py, each atom's channel of largest l local
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import gpu_pseudo_cost as G
    opts = [D.Options(Z, 14, 25.0, 0.0005, 0.5, 0) for Z in range(1, 93)]
    res = ctx.solve_batch(opts, keep_steps=False, radial=True)
    r = res[0].radial.r
    V = np.concatenate([x.radial.V for x in res])
    u, pot, orb, ls, eps, occ, rc = [], [], [], [], [], [], []
    base = 0
    for p, x in enumerate(res):
        u.append(x.radial.orbitals[0])
        for k, l, e, q in G.valence(x):
            pot.append(p); orb.append(base + k); ls.append(l); eps.append(e); occ.append(q)
            rc.append(1.2 * r[G.outermost_extremum(x.radial.orbitals[0][k])])
        base += len(x.radial.orbitals[0])
    grid = (14, 0.0005, 25.0)
    ps = ctx.tm_pseudize(V, np.concatenate(u), *grid, pot, orb, ls, eps, occ, rc)
    pot = np.array(pot)
    keep = np.concatenate([np.nonzero(pot == p)[0] for p in range(len(res)) if np.all(ps.status[pot == p] == 0)])
    idx = {c: k for k, c in enumerate(keep)}
    loc = [idx[keep[(pot[keep] == pot[c]) & (ps.l[keep] == ps.l[pot == pot[c]].max())][0]] for c in keep]
    Vs, us = ps.V_scr[keep], ps.u[keep]
    row, ls, eps = np.arange(len(keep)), ps.l[keep], ps.eps[keep]
    batch = ctx.kb_form(Vs, us, *grid, row, loc, ls, eps)
    E = np.linspace(-2.0, 2.0, 1001)
    ldb = ctx.kb_log_derivatives(batch, Vs, 2.5, E)
    for c in [k for k in (1, len(row) // 2, len(row) - 1) if batch.status[k] != 1] + [int(np.nonzero(batch.status == 1)[0][0])]:
        one = ctx.kb_form(Vs, us, *grid, row[c], loc[c], ls[c], eps[c])
        for f in ("E_KB", "cos", "eps_loc", "r_s", "ghost", "status", "beta"):
            assert np.array_equal(getattr(one, f)[0], getattr(batch, f)[c], equal_nan=True), (c, f)
        ld1 = ctx.kb_log_derivatives(one, Vs, 2.5, E)
        for f in ("D", "u", "du", "nodes"):
            assert np.array_equal(getattr(ld1, f)[0], getattr(ldb, f)[c], equal_nan=True), (c, f)


def test_invalid_arguments_leave_the_outputs_untouched(ctx):
    lib = D.load_library()
    levels, delta, max_r = 12, 0.002, 25.0
    N, r, _, _ = LR.grid(levels, delta, max_r)
    V = np.zeros((2, N))
    V[:, 1:] = -1.0 / np.maximum(r[1:], 0.01)
    V[0, 1:100] -= 0.5
    u = np.stack([r * np.exp(-r), r * np.exp(-r)])
    dp = C.POINTER(C.c_double)

    def form(V=V, u=u, n_rows=2, chans=((0, 1, 0, -0.5),), n_ch=None, grid=(levels, delta, max_r)):
        V = np.ascontiguousarray(V, dtype=np.float64); u = np.ascontiguousarray(u, dtype=np.float64)
        ch = np.zeros(max(1, len(chans)), dtype=np.dtype(_CKbChannel))
        for k, (a, b, l, e) in enumerate(chans):
            ch[k] = (a, b, l, 0, e)
        out = np.zeros(max(1, len(chans)), dtype=np.dtype(_CKbResult)); out["E_KB"] = 7.0
        beta = np.full((max(1, len(chans)), N), 7.0)
        rc = lib.dftatom_kb_form(ctx._h, grid[0], grid[1], grid[2], V.ctypes.data_as(dp), u.ctypes.data_as(dp), n_rows,
                                 ch.ctypes.data_as(C.POINTER(_CKbChannel)), len(chans) if n_ch is None else n_ch,
                                 out.ctypes.data_as(C.POINTER(_CKbResult)), beta.ctypes.data_as(dp))
        return rc, lib.dftatom_last_error().decode(), bool(np.all(out["E_KB"] == 7.0) and np.all(beta == 7.0))

    rc, msg, _ = form()
    assert rc == 0, msg
    bad_V = V.copy(); bad_V[1, 5] = np.nan
    bad_u = u.copy(); bad_u[1, 7] = np.inf
    far = V.copy(); far[0, N - 2] += 1.0
    deep = V.copy(); deep[1, 3] = -118.0 ** 2 - 2.0
    for kw, code, text in [(dict(grid=(0, delta, max_r)), -2, "grid"), (dict(n_rows=0), -5, ""), (dict(n_ch=0), -5, ""),
                           (dict(chans=((2, 1, 0, -0.5),)), -5, "channel 0"), (dict(chans=((0, -1, 0, -0.5),)), -5, "channel 0"),
                           (dict(chans=((0, 1, 4, -0.5),)), -5, "channel 0"), (dict(chans=((0, 1, 0, np.inf),)), -5, "channel 0"),
                           (dict(V=bad_V), -5, "row 1"), (dict(u=bad_u), -5, "row 1"), (dict(V=far), -5, "channel 0"),
                           (dict(V=deep), -5, "too deep")]:
        rc, msg, untouched = form(**kw)
        assert rc == code and text in msg and untouched, (kw, rc, msg)

    beta = np.zeros((1, N)); beta[0, 1:80] = 1.0
    E = np.array([-0.5, 0.1])

    def kbld(V=V, beta=beta, n_proj=1, chans=((1, 0, 0, 1.0, 2.0),), E=E, n_e=None):
        V = np.ascontiguousarray(V, dtype=np.float64); beta = np.ascontiguousarray(beta, dtype=np.float64); E = np.ascontiguousarray(E)
        ch = np.zeros(len(chans), dtype=np.dtype(_CKbLdChannel))
        for k, (p, j, l, ekb, rcut) in enumerate(chans):
            ch[k] = (p, j, l, 0, ekb, rcut)
        out = np.zeros(len(chans) * len(E), dtype=np.dtype(_CLogDeriv)); out["D"] = 7.0
        rc = lib.dftatom_kb_log_derivatives(ctx._h, levels, delta, max_r, V.ctypes.data_as(dp), 2, beta.ctypes.data_as(dp), n_proj,
                                            ch.ctypes.data_as(C.POINTER(_CKbLdChannel)), len(chans), E.ctypes.data_as(dp),
                                            len(E) if n_e is None else n_e, out.ctypes.data_as(C.POINTER(_CLogDeriv)), None)
        return rc, lib.dftatom_last_error().decode(), bool(np.all(out["D"] == 7.0))

    rc, msg, _ = kbld()
    assert rc == 0, msg
    bad_b = beta.copy(); bad_b[0, 3] = np.nan
    far_b = beta.copy(); far_b[0, N - 2] = 1.0
    for kw, text in [(dict(chans=((1, 1, 0, 1.0, 2.0),)), "channel 0"), (dict(chans=((1, -2, 0, 1.0, 2.0),)), "channel 0"),
                     (dict(chans=((1, 0, 0, np.nan, 2.0),)), "channel 0"), (dict(chans=((2, 0, 0, 1.0, 2.0),)), "channel 0"),
                     (dict(chans=((1, 0, 0, 1.0, 0.5 * r[2]),)), "channel 0"), (dict(beta=bad_b), "projector 0"),
                     (dict(beta=far_b), "projector 0"), (dict(E=np.array([0.0, np.nan])), "energy 1"), (dict(V=bad_V), "potential row 1"),
                     (dict(n_proj=-1), ""), (dict(n_e=0), "")]:
        rc, msg, untouched = kbld(**kw)
        assert rc == -5 and text in msg and untouched, (kw, rc, msg)


def test_cli_tables_equal_the_python_calls(ctx):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "bin", "dftatom")
    grid = (14, 0.0005, 25.0)
    with tempfile.TemporaryDirectory() as tmp:
        ps_dir, ld_dir = os.path.join(tmp, "ps"), os.path.join(tmp, "ld")
        subprocess.run([exe, "--Z", "14", "--config", "[Ne] 3s2 3p2 3d0", "--levels", "14", "--delta", "0.0005", "--rmax", "25", "--quiet-steps",
                        "--pseudo", ps_dir, "--pseudo-rc", "2.2,2.0", "--pseudo-local", "2", "--logderiv", ld_dir, "--rc", "2.7",
                        "--energies", "-1:0.5:16"], check=True, capture_output=True, text=True)
        bad = subprocess.run([exe, "--Z", "6", "--levels", "14", "--delta", "0.0005", "--rmax", "25", "--quiet-steps", "--pseudo", ps_dir,
                              "--pseudo-rc", "1.8", "--pseudo-local", "3"], capture_output=True, text=True)
        assert bad.returncode != 0 and "no channel with l = 3" in bad.stderr
        lines = open(os.path.join(ps_dir, "0_Z14_pseudo.tsv")).read().splitlines()
        tab = np.loadtxt(os.path.join(ps_dir, "0_Z14_pseudo.tsv"), delimiter="\t", ndmin=2)
        kbl = open(os.path.join(ld_dir, "0_Z14_pseudo_kb_logderiv.tsv")).read().splitlines()
    heads = [np.array(x[2:].split("\t"), dtype=float) for x in lines[1:4]]
    kbh = [x.split("\t") for x in lines[4:7]]
    assert all(h[0] == "# kb" for h in kbh) and lines[7].startswith("# r\t") and lines[7].endswith("rho_val\tbeta s\tbeta p\tbeta d")
    V_scr, u_ps = tab[:, 4:7].T, tab[:, 7:10].T
    kb = ctx.kb_form(V_scr, u_ps, *grid, [0, 1, 2], 2, [0, 1, 2], [h[2] for h in heads])
    for c, h in enumerate(kbh):
        assert int(h[1]) == c and float(h[2]) == kb.E_KB[c] and float(h[3]) == kb.cos[c]
        assert np.array_equal(np.array(h[4:6], dtype=float), kb.eps_loc[c], equal_nan=True)
        assert int(h[6]) == kb.ghost[c] and int(h[7]) == kb.status[c]
        assert np.array_equal(tab[:, 11 + c], kb.beta[c])
    t = np.loadtxt(kbl[2:], delimiter="\t", ndmin=2)
    E = t[:16, 2]
    got = ctx.kb_log_derivatives(kb, V_scr, 2.7, E)
    assert float(kbl[0].split("r_c=")[1].split()[0]) == got.r_c[0]
    for k in range(3):
        blk = t[16 * k:16 * (k + 1)]
        assert np.all(blk[:, 1] == k) and np.array_equal(blk[:, 3], got.D[k]) and np.array_equal(blk[:, 4], got.nodes[k])
        assert np.array_equal(blk[:, 6], got.u[k]) and np.array_equal(blk[:, 7], got.du[k])
