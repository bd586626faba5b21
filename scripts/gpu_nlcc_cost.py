"""Cost of the nonlinear core correction on the workload of gpu_pseudo_scf_cost.py: C3's atoms (Z = 1..92, 16385 nodes) pseudized at
r_c = 2.5 bohr, solved in the same configurations (reference, cation, s -> p promotion) in one call.  r_pc rule: the outermost node
(1..N-2) where the core density is at least the valence density of the pseudization without a core, kept at r_3 or beyond; an atom
without core levels (H, He) gets the full core (r_pc = 0, rho_pc = 0).
Records the card's name and power limit (read in the same run), the time of one dftatom_partial_core call per atom (host clock around
the synchronous call, median over the atoms and --reps), dftatom_tm_pseudize_core against dftatom_tm_pseudize per atom (alternated,
medians), the device time of the SCF loop (dftatom_last_timing) of the whole batch with and without the core (alternated, --reps each,
after one warm-up of each), and the device time of both instances of pseudo_potential_energy_kernel (torch.profiler trace of a
separate run of each batch).
Usage: python scripts/gpu_nlcc_cost.py --out profiles/r09_nlcc.json"""
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
from gpu_pseudo_cost import LEVELS, DELTA, RMAX, card  # noqa: E402
from gpu_pseudo_scf_cost import R_C, configs  # noqa: E402


def _ms(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def kernel_ms(run):
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as tr:
            run()
            torch.cuda.synchronize()
        ev = [e for e in tr.events() if e.device_time_total > 0 and "pseudo_potential_energy_kernel" in e.name]
        return dict(ms=sum(e.device_time_total for e in ev) / 1e3, launches=len(ev), names=sorted({e.name for e in ev}))
    except Exception as e:          # the trace is a separate measurement: its absence is recorded, not guessed
        return f"not measured ({type(e).__name__})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power, clock = card()
    grid = (LEVELS, DELTA, RMAX)
    with D.Context(0) as ctx:
        res = ctx.solve_batch([D.Options(Z, LEVELS, RMAX, DELTA, 0.5, 0) for Z in range(1, 93)], keep_steps=False, radial=True)
        plain, cored, r_pcs, skipped, t_pc, t_tm, t_tmc = {}, {}, {}, [], [], [], []
        for x in res:
            Z = x.options.Z
            try:
                pp = ctx.pseudize(x, R_C)
            except D.DFTAtomError:
                skipped.append(Z)
                continue
            if np.any(pp.status != 0):
                skipped.append(Z)
                continue
            best = {int(n) * 10 + int(l) for n, l in zip(pp.n, pp.l)}
            core = [k for k, L in enumerate(x.levels[0]) if L.n * 10 + L.l not in best]
            occ = [float(x.levels[0][k].occ) for k in core]
            u = x.radial.orbitals[0]
            r_pc = 0.0
            if core:
                full = ctx.partial_core(u, *grid, 0, core, occ, [0.0])
                rc, rv = full.rho_core[0], pp.rho_val[0]
                hits = [k for k in range(1, len(rc) - 1) if rc[k] >= rv[k]]
                if hits:
                    r_pc = float(pp.r[max(3, max(hits))])
            for _ in range(a.reps):
                t, pc = _ms(lambda: ctx.partial_core(u, *grid, 0, core, occ, [r_pc]))
                t_pc.append(t)
            if pc.status[0] != 0:
                skipped.append(Z)
                continue
            # the pseudization alone, with and without the core, alternated (pseudize's channel choice, as tm_pseudize arguments)
            ls = pp.l.tolist()
            orb = [k for c in range(len(ls)) for k, L in enumerate(x.levels[0]) if (L.n, L.l) == (pp.n[c], ls[c])]
            args = (x.radial.V[0], u, *grid, 0, orb, ls, pp.eps, pp.occ, R_C, pp.n)
            for _ in range(a.reps):
                t, _ = _ms(lambda: ctx.tm_pseudize(*args)); t_tm.append(t)
                t, ppc = _ms(lambda: ctx.tm_pseudize(*args, rho_pc=pc.rho_pc)); t_tmc.append(t)
            plain[Z], cored[Z], r_pcs[Z] = pp, ppc, r_pc
        pps, ppcs, cfgs = [], [], []
        for Z in plain:
            for c in configs(plain[Z]):
                if c is not None:
                    pps.append(plain[Z]); ppcs.append(cored[Z]); cfgs.append(c)
        runs = {"no_core": lambda: ctx.solve_pseudo_batch(pps, cfgs, keep_steps=False),
                "core": lambda: ctx.solve_pseudo_batch(ppcs, cfgs, keep_steps=False)}
        dev, call, out = {k: [] for k in runs}, {k: [] for k in runs}, {}
        for k in runs:
            out[k] = runs[k]()
        for _ in range(a.reps):
            for k in runs:
                t, out[k] = _ms(runs[k])
                call[k].append(t)
                dev[k].append(ctx.last_timing()[0])
        rec = dict(card=name, power_limit=power, max_sm_clock=clock, grid=dict(levels=LEVELS, delta=DELTA, max_r=RMAX, nodes=len(res[0].radial.r)),
                   r_c=R_C, r_pc_rule="outermost node 1..N-2 with rho_core >= rho_val (no core levels: r_pc = 0)", atoms=len(plain),
                   skipped_Z=skipped, r_pc={str(z): v for z, v in r_pcs.items()}, pseudo_atoms=len(cfgs),
                   partial_core_ms_median=float(np.median(t_pc)), tm_pseudize_ms_median=float(np.median(t_tm)),
                   tm_pseudize_core_ms_median=float(np.median(t_tmc)))
        for k in runs:
            rec[k] = dict(device_ms_median=float(np.median(dev[k])), device_ms_all=dev[k], call_ms_median=float(np.median(call[k])),
                          scf_steps_total=int(sum(r.n_steps for r in out[k])),
                          status_counts={str(s): sum(1 for r in out[k] if r.status == s) for s in sorted({r.status for r in out[k]})},
                          kernel9=kernel_ms(runs[k]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps({k: v for k, v in rec.items() if k != "r_pc"}, indent=1))


if __name__ == "__main__":
    main()
