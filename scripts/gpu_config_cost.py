"""Cost of configured atoms on C3 (LDA, 14 levels = 16385 nodes, delta 5e-4, Rmax 25, mixing 0.5): three batches - the 92 neutral atoms,
the cations of Z = 2..92 (H+ has no electron), and both together in one batch.  Records per batch the SCF device time and launches
(dftatom_last_timing), the wall time of solve_batch (median of --reps, batches alternated), the h2d / d2h bytes (dftatom_last_transfer)
and the SCF steps, and from the combined batch the DeltaSCF first ionisation energy E(Z+) - E(Z) of Z = 1..92 (E(H+) = 0).  The card's
name and power limit are read in the same run and stored with the numbers.
Usage: python scripts/gpu_config_cost.py --out profiles/r04_config.json"""
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

LEVELS, DELTA, RMAX, MIX = 14, 0.0005, 25.0, 0.5


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    neutral = [D.Options(Z, LEVELS, RMAX, DELTA, MIX, 0) for Z in range(1, 93)]
    cations = [D.Options(Z, LEVELS, RMAX, DELTA, MIX, 0, charge=1) for Z in range(2, 93)]
    batches = {"neutral": neutral, "cations": cations, "neutral+cations": neutral + cations}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    out = dict(workload="C3 grid: LDA, 14 levels (16385 nodes), delta 0.0005, Rmax 25, mixing 0.5", gpu=smi.strip().splitlines()[0] if smi.strip() else "unknown",
               batches={})
    wall = {k: [] for k in batches}
    with D.Context(0) as ctx:
        for k, opts in batches.items():     # warm-up of every shape
            ctx.solve_batch(opts, keep_steps=False)
        for _ in range(a.reps):             # alternating, so that drifts of the shared host hit every batch alike
            for k, opts in batches.items():
                t0 = time.perf_counter()
                ctx.solve_batch(opts, keep_steps=False)
                wall[k].append((time.perf_counter() - t0) * 1e3)
        res = {}
        for k, opts in batches.items():
            dev = []
            for _ in range(a.reps):
                res[k] = ctx.solve_batch(opts, keep_steps=False)
                dev.append(ctx.last_timing()[0])
            ms, launches = ctx.last_timing()
            h2d, d2h = ctx.last_transfer()
            out["batches"][k] = dict(atoms=len(opts), device_ms_median=float(np.median(dev)), device_ms=dev, wall_ms_median=float(np.median(wall[k])),
                                     wall_ms=wall[k], launches=launches, h2d_bytes=h2d, d2h_bytes=d2h,
                                     scf_steps=sum(r.n_steps for r in res[k]), converged=sum(r.finished for r in res[k]))
    both = res["neutral+cations"]
    e0 = {o.Z: r.Etotal for o, r in zip(neutral, both[:92])}
    e1 = {o.Z: r.Etotal for o, r in zip(cations, both[92:])}
    e1[1] = 0.0
    conv = {o.Z: r.finished for o, r in zip(neutral, both[:92])}
    conv1 = {o.Z: r.finished for o, r in zip(cations, both[92:])}
    conv1[1] = True
    out["first_ionisation_energy_Ha"] = {str(Z): e1[Z] - e0[Z] for Z in range(1, 93)}
    out["ip_both_converged"] = {str(Z): bool(conv[Z] and conv1[Z]) for Z in range(1, 93)}
    out["note"] = ("DeltaSCF first ionisation energy E(Z+) - E(Z) in Hartree (LDA, the reference's Aufbau configurations; cations by "
                   "dftatom_config_aufbau: the electron leaves the occupied subshell of largest n, then l); ip_both_converged: both SCFs met "
                   "the stop test within the 100-step cap (otherwise the energies of the last step)")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(out["gpu"])
    for k, b in out["batches"].items():
        print(f"{k}: {b['atoms']} atoms, device {b['device_ms_median']:.2f} ms, wall {b['wall_ms_median']:.2f} ms, {b['launches']} launches, "
              f"h2d {b['h2d_bytes']} B, {b['scf_steps']} steps, {b['converged']} converged")


if __name__ == "__main__":
    main()
