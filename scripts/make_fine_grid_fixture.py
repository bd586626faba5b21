#!/usr/bin/env python
"""Generate tests/golden/fine_grid.json: the SCF on 18-20-level grids (262145 .. 1048577 nodes) from the C restatement oracle
(oracle/dftatom_oracle.c), for a fixed number of steps.  Test infrastructure only.

usage: python scripts/make_fine_grid_fixture.py [--steps K] [--jobs J]

The unmodified reference is not used here (this fixture is built from the restatement, which tests/test_oracle.py pins on the
reference at smaller grids).  At these sizes the restatement does not fire its own stop test within its step cap (measured: H at 18
levels reaches the 100-step cap, its FP64 multigrid rounding floor keeps |dE/E| above 1e-11), so the fixture holds the first K steps
and the tests compare step by step (run_to_cap, step_cap = K), never stop steps.

Each atom is run twice, with 100 V-cycles per Poisson solve (the reference's setting, the fixture) and with 12: the per-step difference
of the two is recorded as the floor of the oracle's own Poisson solve at that size ("floor_eig", "floor_energy").
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

KEYS = ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc")
G18 = dict(levels=18, delta=5e-5, rmax=50.0, mixing=0.5)
CASES = {
    "H_L18": [dict(Z=1, method=0, **G18)],
    "He_L19": [dict(Z=2, method=0, levels=19, delta=2.5e-5, rmax=50.0, mixing=0.5)],
    "Li_L20": [dict(Z=3, method=1, levels=20, delta=1.25e-5, rmax=50.0, mixing=0.5)],
    # one batch of four: >= 4 atoms put the cold Poisson solves on the stream solver (fewer: one team of CTAs per density)
    "batch_L18": [dict(Z=z, method=m, **G18) for z, m in ((2, 0), (3, 1), (4, 0), (7, 1))],
}


def _run(cfg, steps, max_vcycles):
    """The first `steps` records of the oracle SCF.  orc_scf has no step cap: it runs in a worker process whose step callback
    returns the records through a pipe and ends the process once it has them."""
    import multiprocessing as mp
    rd, wr = mp.Pipe(duplex=False)
    p = mp.get_context("fork").Process(target=_child, args=(cfg, steps, max_vcycles, wr))
    t0 = time.time()
    p.start()
    wr.close()
    recs = rd.recv()
    p.join()
    return recs, time.time() - t0


def _child(cfg, steps, max_vcycles, wr):
    import oracle_lib as O
    out = []

    def cb(st, _):
        s = st.contents
        out.append(dict(E=[s.lv[sp][k].E for sp in range(2) for k in range(s.n_levels[sp])],
                        levels=[(s.lv[sp][k].n0 + 1, s.lv[sp][k].l, s.lv[sp][k].occ) for sp in range(2) for k in range(s.n_levels[sp])],
                        energies=[getattr(s, k) for k in KEYS]))
        if len(out) == steps:
            wr.send(out)
            os._exit(0)

    o = O.OrcOptions(cfg["Z"], cfg["levels"], cfg["rmax"], cfg["delta"], cfg["mixing"], cfg["method"])
    r = O.OrcResult()
    O.oracle().orc_scf(O.C.byref(o), O.C.byref(r), O.STEP_CB(cb), None, max_vcycles)
    wr.send(out)            # (stopped before `steps` steps)
    os._exit(0)


def one(args):
    cfg, steps = args
    recs, sec = _run(cfg, steps, 100)
    floor, sec12 = _run(cfg, steps, 12)
    n = min(len(recs), len(floor))
    return dict(options=cfg, n_steps=len(recs), max_vcycles=100,
                levels=[dict(n=a, l=b, occ=c) for a, b, c in recs[-1]["levels"]],
                eig_per_step=[s["E"] for s in recs], energies_per_step=[s["energies"] for s in recs],
                floor_eig=max(abs(x - y) for k in range(n) for x, y in zip(recs[k]["E"], floor[k]["E"])),
                floor_energy=max(abs(x - y) for k in range(n) for x, y in zip(recs[k]["energies"], floor[k]["energies"])),
                cpu_seconds=round(sec, 1), cpu_seconds_12_vcycles=round(sec12, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--jobs", type=int, default=max(1, (os.cpu_count() or 2) - 1))
    a = ap.parse_args()
    import oracle_lib as O
    O.oracle()                  # (built once, before the workers fork)
    flat = [(name, cfg) for name, cfgs in CASES.items() for cfg in cfgs]
    order = sorted(range(len(flat)), key=lambda i: -flat[i][1]["levels"])        # longest first
    t0 = time.time()
    with ProcessPoolExecutor(a.jobs) as ex:
        res = dict(zip(order, ex.map(one, [(flat[i][1], a.steps) for i in order])))
    out = {name: [] for name in CASES}
    for i, (name, _) in enumerate(flat):
        out[name].append(res[i])
    meta = dict(source="C restatement oracle (oracle/dftatom_oracle.c, orc_scf); the unmodified reference was not run for this fixture",
                steps=a.steps, wall_seconds=round(time.time() - t0, 1), cpu=os.uname().machine)
    path = os.path.join(ROOT, "tests", "golden", "fine_grid.json")
    with open(path, "w") as f:
        json.dump(dict(meta=meta, cases=out), f, indent=1)
    print(json.dumps({k: [(r["options"]["Z"], r["n_steps"], r["cpu_seconds"], r["floor_eig"], r["floor_energy"]) for r in v] for k, v in out.items()}))


if __name__ == "__main__":
    main()
