"""Cost of the Kleinman-Bylander form (dftatom_kb_form) and of its logarithmic derivatives (dftatom_kb_log_derivatives) on C3's
pseudopotentials (16385 nodes, delta 5e-4, Rmax 25): the Aufbau valence channels of Z = 1..92 pseudized as in r06_pseudo.json
(r_c = 1.2 x the radius of the outermost extremum of |u|), the atoms whose channels all succeeded, each with its channel of largest l
as the local potential; then every channel swept over 1001 energies in [-2, 2] at r_c = 2.5 bohr (the radius of r05_logderiv.json).
Records the card's name and power limit, the call times (host clock around the synchronous call, median of --reps after one warm-up
call), the device time per call of the kernels (torch.profiler trace of a separate run), the GSS verdicts, and the lane-node-steps of
the sweep: i_c per lane without projector, max(i_c, i_s) + i_c with one (the driven sweep and the counting pass).
Usage: python scripts/gpu_kb_cost.py --out profiles/r07_kb.json"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import dftatom_b200 as D  # noqa: E402
from gpu_pseudo_cost import LEVELS, DELTA, RMAX, card, outermost_extremum, valence  # noqa: E402

R_C = 2.5


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, [t * 1e3 for t in ts]


def kernel_ms(fn, reps, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_time_total > 0 and "Memcpy" not in e.name and "Memset" not in e.name]
    if not ev:
        return None
    out = {f"{k}_ms_per_call": sum(e.device_time_total for e in ev if k in e.name) / 1e3 / reps for k in names}
    out["all_kernels_ms_per_call"] = sum(e.device_time_total for e in ev) / 1e3 / reps
    out["kernels"] = sorted({e.name for e in ev})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power, clock = card()
    with D.Context(0) as ctx:
        res = ctx.solve_batch([D.Options(Z, LEVELS, RMAX, DELTA, 0.5, 0) for Z in range(1, 93)], keep_steps=False, radial=True)
        r = res[0].radial.r
        V = np.concatenate([x.radial.V for x in res])
        u, pot, orb, ls, eps, occ, rc = [], [], [], [], [], [], []
        base = 0
        for p, x in enumerate(res):
            u.append(x.radial.orbitals[0])
            for k, l, e, q in valence(x):
                pot.append(p); orb.append(base + k); ls.append(l); eps.append(e); occ.append(q)
                rc.append(1.2 * r[outermost_extremum(x.radial.orbitals[0][k])])
            base += len(x.radial.orbitals[0])
        ps = ctx.tm_pseudize(V, np.concatenate(u), LEVELS, DELTA, RMAX, pot, orb, ls, eps, occ, rc)
        pot = np.array(pot)
        good = [p for p in range(len(res)) if np.all(ps.status[pot == p] == 0)]
        keep = np.concatenate([np.nonzero(pot == p)[0] for p in good])
        loc = np.array([keep[(pot[keep] == pot[c]) & (ps.l[keep] == ps.l[pot == pot[c]].max())][0] for c in keep])
        idx = {c: k for k, c in enumerate(keep)}
        Vs, us = ps.V_scr[keep], ps.u[keep]
        args = (Vs, us, LEVELS, DELTA, RMAX, np.arange(len(keep)), [idx[c] for c in loc], ps.l[keep], ps.eps[keep])
        kb = ctx.kb_form(*args)
        E = np.linspace(-2.0, 2.0, 1001)
        ld = ctx.kb_log_derivatives(kb, Vs, R_C, E)
        ic = LR_nearest(r, R_C)
        steps = sum((ic if kb.status[c] == 1 else max(ic, int(kb.i_s[c])) + ic) for c in range(len(keep))) * len(E)
        rec = dict(card=name, power_limit=power, max_sm_clock=clock, grid=dict(levels=LEVELS, delta=DELTA, max_r=RMAX, nodes=len(r)),
                   atoms=len(good), channels=int(len(keep)), local_channels=int(np.sum(kb.status == 1)),
                   status_counts={str(s): int(np.sum(kb.status == s)) for s in np.unique(kb.status)},
                   ghosts=int(np.sum(kb.ghost == 1)), energies=len(E), r_c=R_C, lane_node_steps=float(steps),
                   nan_lanes=int(np.sum(ld.nodes < 0)))
        t, ts = timed(lambda: ctx.kb_form(*args), a.reps)
        rec["kb_form"] = dict(call_ms_median=t, call_ms_all=ts, kernels=kernel_ms(lambda: ctx.kb_form(*args), a.reps, ["kb_form_kernel"]) or "not measured")
        t, ts = timed(lambda: ctx.kb_log_derivatives(kb, Vs, R_C, E), a.reps)
        km = kernel_ms(lambda: ctx.kb_log_derivatives(kb, Vs, R_C, E), a.reps, ["kb_logderiv_kernel", "kb_proj_kernel"])
        rec["kb_log_derivatives"] = dict(call_ms_median=t, call_ms_all=ts, kernels=km or "not measured")
        if km:
            rec["kb_log_derivatives"]["lane_node_steps_per_s"] = steps / (km["kb_logderiv_kernel_ms_per_call"] * 1e-3)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


def LR_nearest(r, r_c):
    N = len(r)
    hi = int(np.searchsorted(r[2:N - 1], r_c, side="left")) + 2
    return hi - 1 if hi > 2 and r_c - r[hi - 1] <= r[hi] - r_c else hi


if __name__ == "__main__":
    main()
