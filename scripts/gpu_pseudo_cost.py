"""Cost of the Troullier-Martins pseudization and unscreening (dftatom_tm_pseudize) on two workloads (16385 nodes, delta 5e-4, Rmax 25):
  C3     the Aufbau valence channels of Z = 1..92 (LDA; the level of largest n for every l), r_c = 1.2 x the radius of the outermost
         extremum of |u|; every atom is one potential row, so the call also runs 92 valence densities, Poisson solves and unscreenings
  Si-rc  Si [Ne] 3s2 3p2 3d0, 3 channels (3s, 3p, 3d) at each of 64 radii in [1.4, 3.0] bohr: 64 potential rows of 3 channels
Records the card's name and power limit, the call time (host clock around the synchronous call, median of --reps after one warm-up
call), and the device time per call of the kernels (torch.profiler trace of a separate run): tm_kernel alone and all kernels of the
call (tm_kernel, the a-table, the density, the cold Poisson solve, VWN and the unscreening), with the channels' statuses.
Usage: python scripts/gpu_pseudo_cost.py --out profiles/r06_pseudo.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dftatom_b200 as D  # noqa: E402

LEVELS, DELTA, RMAX = 14, 0.0005, 25.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
        return [x.strip() for x in q.split(",")]
    except (OSError, subprocess.CalledProcessError, IndexError):
        return ["not measured"] * 3


def valence(res):
    """(orbital row, l, eps, occ) of the level of largest n for every l of levels[0]."""
    best = {}
    for k, lev in enumerate(res.levels[0]):
        if lev.l not in best or lev.n > res.levels[0][best[lev.l]].n:
            best[lev.l] = k
    return [(best[l], l, res.levels[0][best[l]].E, float(res.levels[0][best[l]].occ)) for l in sorted(best)]


def outermost_extremum(u):
    """Node of the largest |u| beyond the last sign change."""
    sgn = np.sign(u[1:])
    flips = np.nonzero(sgn[1:] * sgn[:-1] < 0)[0]
    i0 = flips[-1] + 2 if len(flips) else 1
    return i0 + int(np.argmax(np.abs(u[i0:])))


def timed(ctx, args, reps):
    ctx.tm_pseudize(*args)                          # warm-up: grid tables, scratch buffers, module load
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = ctx.tm_pseudize(*args)
        ts.append(time.perf_counter() - t0)
    return out, float(np.median(ts)), [t * 1e3 for t in ts]


def kernel_ms(ctx, args, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.tm_pseudize(*args)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_time_total > 0 and "Memcpy" not in e.name and "Memset" not in e.name]
    if not ev:
        return None
    tm = sum(e.device_time_total for e in ev if "tm_kernel" in e.name) / 1e3 / reps
    total = sum(e.device_time_total for e in ev) / 1e3 / reps
    names = sorted({e.name for e in ev})
    return dict(tm_kernel_ms_per_call=tm, all_kernels_ms_per_call=total, kernels=names)


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
        u = np.concatenate(u)
        si = ctx.solve_batch([D.Options(14, LEVELS, RMAX, DELTA, 0.5, 0, config="[Ne] 3s2 3p2 3d0")], keep_steps=False, radial=True)[0]
        sch = valence(si)
        radii = np.linspace(1.4, 3.0, 64)
        setups = {
            "C3": (V, u, LEVELS, DELTA, RMAX, pot, orb, ls, eps, occ, rc),
            "Si-rc": (np.repeat(si.radial.V[0][None, :], 64, axis=0), si.radial.orbitals[0], LEVELS, DELTA, RMAX, np.repeat(np.arange(64), 3),
                      np.tile([c[0] for c in sch], 64), np.tile([c[1] for c in sch], 64), np.tile([c[2] for c in sch], 64),
                      np.tile([c[3] for c in sch], 64), np.repeat(radii, 3)),
        }
        rec = dict(card=name, power_limit=power, max_sm_clock=clock, grid=dict(levels=LEVELS, delta=DELTA, max_r=RMAX, nodes=len(r)), cases={})
        for key, args in setups.items():
            out, t, ts = timed(ctx, args, a.reps)
            km = kernel_ms(ctx, args, a.reps)
            rec["cases"][key] = dict(channels=int(len(out.l)), potential_rows=int(out.rho_val.shape[0]),
                                     status_counts={str(s): int(np.sum(out.status == s)) for s in np.unique(out.status)},
                                     call_ms_median=t * 1e3, call_ms_all=ts,
                                     kernels=km if km is not None else "not measured")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
