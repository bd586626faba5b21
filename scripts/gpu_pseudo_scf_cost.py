"""Cost of the self-consistent pseudo-atom (dftatom_solve_pseudo_batch) on C3's atoms (Z = 1..92, 16385 nodes, delta 5e-4, Rmax 25):
every atom pseudized with r_c = 2.5 bohr on all its valence channels (the radius of r07_kb.json; atoms whose pseudization fails are
left out and counted), then every atom solved in three configurations in one call: the reference valence configuration, the +1
cation (one electron less in the channel of highest eigenvalue, where the valence charge stays above 0) and an s -> p promotion (where
the atom has both channels, an s electron and room in p).  Records the card's name and power limit, the call time (host clock around
the synchronous call) and the device time of the SCF loop (dftatom_last_timing), medians of --reps after one warm-up call, the SCF
steps and kernel launches, the search rounds per orbital solve (set_option "profile", a separate call), and the device time of
pseudo_potential_energy_kernel (torch.profiler trace of a separate run).
Usage: python scripts/gpu_pseudo_scf_cost.py --out profiles/r08_pseudo_scf.json"""
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

R_C = 2.5


def configs(pp):
    """(reference, cation or None, promotion or None) as (n, l, occ) entry lists."""
    ref = [(int(n), int(l), float(q)) for n, l, q in zip(pp.n, pp.l, pp.occ)]
    Q = sum(q for _, _, q in ref)
    cat = None
    occd = [k for k, e in enumerate(ref) if e[2] >= 1.0]
    if Q - 1.0 > 0 and occd:
        k = max(occd, key=lambda k: pp.eps[k])
        cat = [e if j != k else (e[0], e[1], e[2] - 1.0) for j, e in enumerate(ref)]
    pro = None
    s = [k for k, e in enumerate(ref) if e[1] == 0]
    p = [k for k, e in enumerate(ref) if e[1] == 1]
    if s and p and ref[s[0]][2] >= 1.0 and ref[p[0]][2] <= 5.0:
        pro = [(e[0], e[1], e[2] - 1.0) if j == s[0] else ((e[0], e[1], e[2] + 1.0) if j == p[0] else e) for j, e in enumerate(ref)]
    return ref, cat, pro


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power, clock = card()
    with D.Context(0) as ctx:
        res = ctx.solve_batch([D.Options(Z, LEVELS, RMAX, DELTA, 0.5, 0) for Z in range(1, 93)], keep_steps=False, radial=True)
        pps, cfgs, kinds, skipped = [], [], [], []
        for x in res:
            try:
                pp = ctx.pseudize(x, R_C)
            except D.DFTAtomError:
                skipped.append(x.options.Z)
                continue
            if np.any(pp.status != 0):
                skipped.append(x.options.Z)
                continue
            for kind, c in zip(("reference", "cation", "promotion"), configs(pp)):
                if c is not None:
                    pps.append(pp); cfgs.append(c); kinds.append(kind)
        run = lambda: ctx.solve_pseudo_batch(pps, cfgs, keep_steps=False)
        out = run()
        call, dev = [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            out = run()
            call.append((time.perf_counter() - t0) * 1e3)
            dev.append(ctx.last_timing()[0])
        launches = ctx.last_timing()[1]
        ctx.set_option("profile", 1)
        try:
            run()
            prof = ctx.last_profile()
        finally:
            ctx.set_option("profile", 0)
        rec = dict(card=name, power_limit=power, max_sm_clock=clock, grid=dict(levels=LEVELS, delta=DELTA, max_r=RMAX, nodes=len(res[0].radial.r)),
                   r_c=R_C, atoms=len(res) - len(skipped), skipped_Z=skipped, pseudo_atoms=len(out),
                   configurations={k: kinds.count(k) for k in ("reference", "cation", "promotion")},
                   status_counts={str(s): sum(1 for r in out if r.status == s) for s in sorted({r.status for r in out})},
                   scf_steps_total=int(sum(r.n_steps for r in out)), scf_steps_max=int(max(r.n_steps for r in out)),
                   launches=int(launches), call_ms_median=float(np.median(call)), call_ms_all=call,
                   device_ms_median=float(np.median(dev)), device_ms_all=dev,
                   orbital_solves=prof["match"]["work"], search_rounds=prof["density"]["work"],
                   search_rounds_per_solve=prof["density"]["work"] / max(1.0, prof["match"]["work"]))
        try:
            import torch
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.init()
            with profile(activities=[ProfilerActivity.CUDA]) as tr:
                run()
                torch.cuda.synchronize()
            ev = [e for e in tr.events() if e.device_time_total > 0]
            rec["pseudo_potential_energy_kernel_ms"] = sum(e.device_time_total for e in ev if "pseudo_potential_energy_kernel" in e.name) / 1e3
            rec["pseudo_potential_energy_kernel_launches"] = sum(1 for e in ev if "pseudo_potential_energy_kernel" in e.name)
            rec["all_kernels_ms"] = sum(e.device_time_total for e in ev if "Memcpy" not in e.name and "Memset" not in e.name) / 1e3
        except Exception as e:      # the trace is a separate measurement: its absence is recorded, not guessed
            rec["pseudo_potential_energy_kernel_ms"] = f"not measured ({type(e).__name__})"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
