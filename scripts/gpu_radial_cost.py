"""Cost of the radial export on C3 (Z = 1..92, LDA, 16385 nodes, delta 5e-4, Rmax 25): the sweep with the export off, with the fields only
(rho, V, V_H, electron counts) and with fields plus orbitals and their moments.  Records per mode the wall time of solve_batch (median of
--reps, modes alternated), the SCF device time and launches (dftatom_last_timing, which excludes the export), the d2h bytes
(dftatom_last_transfer), and the export's wall time (the mode's median minus that of "off").  For the split between the export kernels
and the copies: the time of one device -> host copy of the same byte count into pageable and into pinned memory (torch, CUDA events
around a copy that ends in a synchronise).  The card's name and power limit are recorded with the numbers.
Usage: python scripts/gpu_radial_cost.py --out profiles/r03_radial.json"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dftatom_b200 as D  # noqa: E402
from dftatom_b200.api import _COptions, _CRadial, _CResult, _check  # noqa: E402

LEVELS, DELTA, RMAX = 14, 0.0005, 25.0


def solve(ctx, copts, n, cres, arrays, mode):
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    if mode == "off":
        return _check(ctx._lib.dftatom_solve_batch(ctx._h, copts, n, cres, None, 0))
    r, rho, v, vh, am, orb, mom = arrays
    full = mode == "fields+orbitals"
    rad = _CRadial(p(r), p(rho), p(v), p(vh), p(orb) if full else None, orb.shape[0], p(mom) if full else None, p(am))
    return _check(ctx._lib.dftatom_solve_batch_radial(ctx._h, copts, n, cres, None, 0, C.byref(rad)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch

    opts = [D.Options(Z, LEVELS, RMAX, DELTA, 0.5, 0) for Z in range(1, 93)]
    n, N = len(opts), D.n_nodes(LEVELS)
    rows = sum(D.orbital_count(o.Z, o.method) for o in opts)
    arrays = (np.zeros(N), np.zeros((n, 2, N)), np.zeros((n, 2, N)), np.zeros((n, N)), np.zeros((n, 2)), np.zeros((rows, N)),
              np.zeros((rows, D.api.N_MOMENTS)))
    copts = (_COptions * n)(*[o._c() for o in opts])
    cres = (_CResult * n)()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    out = dict(workload="C3: Z = 1..92, LDA, 14 levels (16385 nodes), delta 0.0005, Rmax 25, mixing 0.5", atoms=n, orbital_rows=rows, nodes=N,
               orbital_bytes=rows * N * 8, gpu=smi.strip().splitlines()[0] if smi.strip() else "unknown", modes={})
    modes = ("off", "fields", "fields+orbitals")
    with D.Context(0) as ctx:
        for m in modes:                     # warm-up of every shape, host arrays touched once
            solve(ctx, copts, n, cres, arrays, m)
        wall = {m: [] for m in modes}
        for _ in range(a.reps):             # alternating, so that drifts of the shared host hit every mode alike
            for m in modes:
                t0 = time.perf_counter()
                solve(ctx, copts, n, cres, arrays, m)
                wall[m].append((time.perf_counter() - t0) * 1e3)
            print("rep done", flush=True)
        for m in modes:
            solve(ctx, copts, n, cres, arrays, m)
            ms, launches = ctx.last_timing()
            h2d, d2h = ctx.last_transfer()
            out["modes"][m] = dict(wall_ms_median=float(np.median(wall[m])), wall_ms=wall[m], scf_device_ms=ms, scf_launches=launches, h2d_bytes=h2d,
                                   d2h_bytes=d2h)
    out["export_wall_ms"] = {m: out["modes"][m]["wall_ms_median"] - out["modes"]["off"]["wall_ms_median"] for m in modes[1:]}
    out["export_d2h_bytes"] = {m: out["modes"][m]["d2h_bytes"] - out["modes"]["off"]["d2h_bytes"] for m in modes[1:]}
    copy = {}
    for m in modes[1:]:
        nb = out["export_d2h_bytes"][m]
        src = torch.empty(nb // 8, dtype=torch.float64, device="cuda")
        for kind, dst in (("pageable", torch.empty(nb // 8, dtype=torch.float64)), ("pinned", torch.empty(nb // 8, dtype=torch.float64).pin_memory())):
            t = []
            for _ in range(a.reps + 1):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                dst.copy_(src)
                e1.record()
                torch.cuda.synchronize()
                t.append(e0.elapsed_time(e1))
            copy[f"{m}:{kind}"] = dict(bytes=nb, ms_median=float(np.median(t[1:])), GBps=nb / (np.median(t[1:]) * 1e-3) / 1e9)
        del src
    out["d2h_copy_same_bytes"] = copy
    out["note"] = ("export_wall_ms: extra wall time of solve_batch with the export (kernels + copies into the caller's pageable arrays); "
                   "d2h_copy_same_bytes: one copy of the export's byte count, to split that time between the copies and the kernels")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "modes"}))
    for m in modes:
        r = out["modes"][m]
        print(m, "wall %.2f ms, SCF %.2f ms, %d launches, d2h %d B" % (r["wall_ms_median"], r["scf_device_ms"], r["scf_launches"], r["d2h_bytes"]))
    print(json.dumps(copy))


if __name__ == "__main__":
    main()
