"""numpy / scipy reference of the self-consistent pseudo-atom of dftatom_solve_pseudo_batch (definition: include/dftatom_b200.h).
Every step runs the all-electron loop in its order: each entry's eigenvalue with n - n_ref nodes in its V_l,s (the node-count
bisection of kb_ref.local_levels on the bracket [-Z_b^2 - 1, 50], counted by the engine's Sturm predicate in the oracle's C sweep for
speed), its matched and normalised Numerov orbital (the oracle), the density and its linear mixing, U from the banded solve of
pseudo_ref.hartree_U, the VWN LDA / LSDA of the oracle, and the energies and stop test of the definition."""
import numpy as np

import kb_ref as KB
import oracle_lib as O
import pseudo_ref as P

STOP_TOL = 1e-11          # |dE / E| of the all-electron stop test


def z_bracket(v_ion_rows):
    """Z_b: the smallest integer >= 1 with -Z_b^2 - 1 <= min V_ion - 10 over nodes 1..N-1 of the atom's channels."""
    vmin = min(float(np.min(v[1:])) for v in v_ion_rows)
    z = 1
    while -float(z * z) - 1.0 > vmin - 10.0:
        z += 1
    return z


def level(V, delta, max_r, l, nodes, zb, tol=1e-14):
    """The eigenvalue with `nodes` nodes: bisection on the count of sign changes (> nodes: above the level)."""
    lo, hi = -float(zb * zb) - 1.0, 50.0
    while hi - lo > tol * max(1.0, abs(lo)):
        mid = 0.5 * (lo + hi)
        if O.numerov_count_all(V, delta, max_r, [l], [mid])[0] > nodes:
            hi = mid
        else:
            lo = mid
    return lo


def solve(v_ion, n_ref, config, levels, delta, max_r, mixing=0.5, method=0, max_steps=None):
    """v_ion: {l: V_ion row [N]}, n_ref: {l: n}, config: (n, l, spin, occ) entries.  Returns dict(E [[per spin, (n, l) order]],
    levels [[(n, l, occ)]], Etotal, Ekin, Ecoul, Eenuc, Exc, n_steps, converged, u [[orbital rows]], rho [n_spin][N], v [n_spin][N]
    (the screening V_H + V_xc), steps [dicts])."""
    N, r, K, jac, sqex, wjac = KB.tables(levels, delta, max_r)
    ns = 2 if method & 1 else 1
    inv4pr2 = np.zeros(N)
    inv4pr2[1:] = 1.0 / (4 * np.pi * r[1:] ** 2)
    ent = [sorted([e for e in config if e[2] == s], key=lambda e: (e[0], e[1])) for s in range(ns)]
    n_el = [sum(e[3] for e in ent[s]) for s in range(ns)]
    Q = sum(n_el)
    zb = z_bracket([v_ion[l] for l in v_ion])
    cap = max_steps or (150 if ns == 2 else 100)
    volume = 4 * np.pi / 3 * max_r ** 3
    rho = [np.where(np.arange(N) == 0, 0.0, n_el[s] / volume) for s in range(ns)]

    def potential(rho):
        rt = rho[0] + rho[1] if ns == 2 else rho[0]
        U = P.hartree_U(levels, delta, max_r, rt, Q)
        if ns == 2:
            va, vb, vexc, edif = O.vwn_lsda(rho[0], rho[1])
            vxc = [va, vb]
        else:
            vexc, edif = O.vwn_lda(rho[0])
            vxc = [vexc]
        S = []
        for s in range(ns):
            x = np.zeros(N)
            x[1:] = U[1:] / r[1:] + vxc[s][1:]
            S.append(x)
        return rt, U, S, vexc, edif

    rt, U, S, vexc, edif = potential(rho)
    e_old, prev_ok, steps = 0.0, False, []
    converged = False
    for step in range(cap):
        V = {(s, l): v_ion[l] + S[s] for s in range(ns) for l in v_ion}
        E, u = [], []
        for s in range(ns):
            E.append([]); u.append([])
            for n, l, _, occ in ent[s]:
                eps = level(V[(s, l)], delta, max_r, l, n - n_ref[l], zb)
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
        rt, U, S, vexc, edif = potential(rho)
        i = slice(1, N)
        rd = r[i] * rt[i] * wjac[i]
        e_dif = 4 * np.pi * np.sum(r[i] * rd * edif[i])
        e_xc = 4 * np.pi * np.sum(r[i] * rd * vexc[i]) + e_dif
        e_h = 0.5 * 4 * np.pi * np.sum(rd * U[i])
        e_ion = e_pot = 0.0
        for s in range(ns):
            for k, (n, l, _, occ) in enumerate(ent[s]):
                w = occ * wjac[i] * u[s][k][i] ** 2
                e_ion += np.sum(w * v_ion[l][i])
                e_pot += np.sum(w * (v_ion[l][i] + S[s][i]))
        etot = eel - e_h + e_dif
        rec = dict(E=E, Etotal=etot, Ekin=eel - e_pot, Ecoul=e_h, Eenuc=e_ion, Exc=e_xc)
        steps.append(rec)
        crit = abs((e_old - etot) / etot) < STOP_TOL and prev_ok
        e_old, prev_ok = etot, True
        if crit:
            converged = True
            break
    last = steps[-1]
    return dict(last, levels=[[(e[0], e[1], e[3]) for e in ent[s]] for s in range(ns)], n_steps=len(steps), converged=converged, u=u,
                rho=rho, v=S, steps=steps, z_b=zb)
