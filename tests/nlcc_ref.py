"""numpy / scipy reference of the nonlinear core correction (definitions: dftatom_partial_core, dftatom_tm_pseudize_core and
dftatom_solve_pseudo_batch_core in include/dftatom_b200.h): the core density, the Louie-Froyen-Cohen partial core (root by
scipy.optimize.brentq), the core-corrected unscreening with the pieces of pseudo_ref, and the core-corrected pseudo-atom SCF with the
helpers of pseudo_scf_ref (which stays as it is)."""
import numpy as np
from scipy.optimize import brentq

import kb_ref as KB
import logderiv_ref as LR
import oracle_lib as O
import pseudo_ref as P
import pseudo_scf_ref as PS


def core_density(u_rows, occ, levels, delta, max_r):
    """sum occ u^2 / (4 pi r^2) at nodes 1..N-2, 0 at nodes 0 and N-1."""
    N, r, _, _ = LR.grid(levels, delta, max_r)
    rho = np.zeros(N)
    for u, o in zip(u_rows, occ):
        rho[1:N - 1] += o * np.asarray(u, np.float64)[1:N - 1] ** 2
    rho[1:N - 1] /= 4 * np.pi * r[1:N - 1] ** 2
    return rho


def partial_core(rho_core, levels, delta, max_r, r_pc):
    """dict(r_pc, i_pc, A, B, t, status, rho_pc, n_core, n_pc)."""
    N, r, _, _, _, wjac = KB.tables(levels, delta, max_r)
    w = wjac * 4 * np.pi * r * r
    out = dict(n_core=float(np.sum(w * rho_core)))
    if r_pc == 0.0:
        return dict(out, r_pc=0.0, i_pc=0, A=0.0, B=0.0, t=np.nan, status=0, rho_pc=rho_core.copy(), n_pc=out["n_core"])
    n = LR.nearest_node(r, r_pc)
    rc = r[n]
    rho = rho_core[n]
    di = ((rho_core[n - 2] - 8 * rho_core[n - 1]) + (8 * rho_core[n + 1] - rho_core[n + 2])) / 12
    J = max_r / (N - 1) if delta == 0.0 else delta * (rc + max_r / (np.exp((N - 1) * delta) - 1.0))
    t = 1 + rc * (di / J) / rho if rho > 0 else np.nan
    if not (rho > 0 and t < 1):
        bad = np.full(N, np.nan)
        bad[0] = 0.0
        return dict(out, r_pc=rc, i_pc=n, A=np.nan, B=np.nan, t=t, status=1, rho_pc=bad, n_pc=np.nan)
    x = brentq(lambda x: x * np.cos(x) - t * np.sin(x), 1e-300, np.pi, xtol=1e-300, rtol=8.9e-16, maxiter=500)
    B, A = x / rc, rho * rc / np.sin(x)
    pc = rho_core.copy()
    pc[0] = 0.0
    pc[1:n] = A * np.sin(B * r[1:n]) / r[1:n]
    return dict(out, r_pc=rc, i_pc=n, A=A, B=B, t=t, status=0, rho_pc=pc, n_pc=float(np.sum(w * pc)))


def unscreen_core(levels, delta, max_r, channels, rho_pc):
    """pseudo_ref.unscreen with V_xc of rho_val + rho_pc (V_H of rho_val): (rho_v, V_H, V_xc, [V_ion per channel])."""
    N, r, _, _ = LR.grid(levels, delta, max_r)
    if any(ch["status"] for ch, _, _ in channels):
        return P.unscreen(levels, delta, max_r, channels)
    rho, vh, _, _ = P.unscreen(levels, delta, max_r, channels)
    vxc = P.vwn_lda(rho + rho_pc)
    vion = []
    for ch, _, _ in channels:
        v = ch["v_scr"] - vh - vxc
        v[0] = 0.0
        vion.append(v)
    return rho, vh, vxc, vion


def solve(v_ion, n_ref, config, levels, delta, max_r, rho_pc, mixing=0.5, method=0, max_steps=None):
    """pseudo_scf_ref.solve of the core-corrected definition: V_xc,s of rho_s + rho_pc / 2 (LDA: rho + rho_pc), Exc and Etotal with the
    core.  Same return value."""
    N, r, K, jac, sqex, wjac = KB.tables(levels, delta, max_r)
    ns = 2 if method & 1 else 1
    inv4pr2 = np.zeros(N)
    inv4pr2[1:] = 1.0 / (4 * np.pi * r[1:] ** 2)
    ent = [sorted([e for e in config if e[2] == s], key=lambda e: (e[0], e[1])) for s in range(ns)]
    n_el = [sum(e[3] for e in ent[s]) for s in range(ns)]
    Q = sum(n_el)
    zb = PS.z_bracket([v_ion[l] for l in v_ion])
    cap = max_steps or (150 if ns == 2 else 100)
    volume = 4 * np.pi / 3 * max_r ** 3
    rho = [np.where(np.arange(N) == 0, 0.0, n_el[s] / volume) for s in range(ns)]
    pc = np.asarray(rho_pc, np.float64)

    def potential(rho):
        rt = rho[0] + rho[1] if ns == 2 else rho[0]
        U = P.hartree_U(levels, delta, max_r, rt, Q)
        if ns == 2:
            va, vb, vexc, edif = O.vwn_lsda(rho[0] + 0.5 * pc, rho[1] + 0.5 * pc)
            vxc = [va, vb]
            sv = rho[0] * va + rho[1] * vb
        else:
            vexc, edif = O.vwn_lda(rho[0] + pc)
            vxc = [vexc]
            sv = rho[0] * vexc
        S = []
        for s in range(ns):
            x = np.zeros(N)
            x[1:] = U[1:] / r[1:] + vxc[s][1:]
            S.append(x)
        return rt, U, S, np.asarray(vexc) + np.asarray(edif), sv

    rt, U, S, exc, sv = potential(rho)
    e_old, prev_ok, steps = 0.0, False, []
    converged = False
    for step in range(cap):
        V = {(s, l): v_ion[l] + S[s] for s in range(ns) for l in v_ion}
        E, u = [], []
        for s in range(ns):
            E.append([]); u.append([])
            for n, l, _, occ in ent[s]:
                eps = PS.level(V[(s, l)], delta, max_r, l, n - n_ref[l], zb)
                psi, _ = O.orbital(V[(s, l)], delta, max_r, l, eps)
                E[s].append(eps); u[s].append(psi)
        eel = sum(e[3] * E[s][k] for s in range(ns) for k, e in enumerate(ent[s]))
        for s in range(ns):
            acc = np.zeros(N)
            for k, e in enumerate(ent[s]):
                acc[:N - 1] += e[3] * u[s][k][:N - 1] ** 2
            new = rho[s].copy()
            new[1:] = mixing * rho[s][1:] + (1 - mixing) * (acc[1:] * inv4pr2[1:])
            rho[s] = new
        rt, U, S, exc, sv = potential(rho)
        i = slice(1, N)
        w = 4 * np.pi * r[i] ** 2 * wjac[i]
        e_xc = np.sum(w * (rt[i] + pc[i]) * exc[i])
        e_h = 0.5 * 4 * np.pi * np.sum(r[i] * rt[i] * wjac[i] * U[i])
        e_ion = e_pot = 0.0
        for s in range(ns):
            for k, (n, l, _, occ) in enumerate(ent[s]):
                ww = occ * wjac[i] * u[s][k][i] ** 2
                e_ion += np.sum(ww * v_ion[l][i])
                e_pot += np.sum(ww * (v_ion[l][i] + S[s][i]))
        etot = eel - e_h - np.sum(w * sv[i]) + e_xc
        rec = dict(E=E, Etotal=etot, Ekin=eel - e_pot, Ecoul=e_h, Eenuc=e_ion, Exc=e_xc)
        steps.append(rec)
        crit = abs((e_old - etot) / etot) < PS.STOP_TOL and prev_ok
        e_old, prev_ok = etot, True
        if crit:
            converged = True
            break
    last = steps[-1]
    return dict(last, levels=[[(e[0], e[1], e[3]) for e in ent[s]] for s in range(ns)], n_steps=len(steps), converged=converged, u=u,
                rho=rho, v=S, steps=steps, z_b=zb)
