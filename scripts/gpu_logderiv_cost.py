"""Cost of the logarithmic derivatives (dftatom_log_derivatives) on C3 (Z = 1..92, LDA, 16385 nodes, delta 5e-4, Rmax 25): every atom's
converged V, l = 0..3, 1001 energies in [-2, 2], r_c = 2.5 bohr (368 channels, 368368 lanes); and on Ar alone (4 channels x 301
energies).  Records the card's name and power limit, the end-to-end call time (host clock around the synchronous call, median of
--reps after one warm-up call), the kernel time (logderiv_kernel in a torch.profiler trace of a separate run), lane-node-steps per
second, the FP64 instructions per node-step of the sweep loop counted from the library's SASS, and the share of the FP64 issue rate
that dftatom_measure_fp64_peak measures (peak TFLOP/s / 2 = DFMA per second).
Usage: python scripts/gpu_logderiv_cost.py --out profiles/r05_logderiv.json"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dftatom_b200 as D  # noqa: E402

LEVELS, DELTA, RMAX = 14, 0.0005, 25.0
FP64 = re.compile(r"^(@!?U?P\w+\s+)?(DFMA|DMUL|DADD|DSETP|DMNMX|MUFU\.RCP64H|MUFU\.RSQ64H|F2F\.F64|F2F\.F32\.F64|I2F\.F64)\b")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
        return [x.strip() for x in q.split(",")]
    except (OSError, subprocess.CalledProcessError, IndexError):
        return ["not measured"] * 3


def loop_fp64_per_node():
    """FP64 instructions per node-step of logderiv_kernel's main loop (the longest backward branch): FP64 instructions in the loop body
    over the divisions in it (one per node: MUFU.RCP64H starts each)."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        return None
    sass = subprocess.run([cuobjdump, "-sass", "-fun", "_ZN3dft15logderiv_kernelENS_7GridDevENS_12LogDerivArgsE", D.lib_path()],
                          capture_output=True, text=True, check=True).stdout
    ins = []
    for ln in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", ln)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    at = {a: k for k, (a, _) in enumerate(ins)}
    best = None
    for k, (a, t) in enumerate(ins):
        m = re.search(r"BRA\b.*?0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) < a and int(m.group(1), 16) in at:
            body = [x for _, x in ins[at[int(m.group(1), 16)]:k + 1]]
            if best is None or len(body) > len(best):
                best = body
    if not best:
        return None
    fp = sum(1 for x in best if FP64.match(x))
    nodes = sum(1 for x in best if "MUFU.RCP64H" in x)
    return dict(loop_instructions=len(best), loop_fp64_instructions=fp, nodes_per_iteration=nodes,
                fp64_per_node_step=fp / nodes if nodes else None)


def node_steps(r_used, r, n_energies):
    ic = np.array([int(np.argmin(np.abs(r - x))) for x in r_used])
    return float(np.sum(ic) * n_energies)          # nodes 2 .. i_c + 1 per lane


def case(ctx, V, pot, l, r_c, E, reps):
    ctx.log_derivatives(V, LEVELS, DELTA, RMAX, pot, l, r_c, E)     # warm-up: grid tables, scratch buffers, module load
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = ctx.log_derivatives(V, LEVELS, DELTA, RMAX, pot, l, r_c, E)
        ts.append(time.perf_counter() - t0)
    return out, float(np.median(ts)), [float(t) for t in ts]


def kernel_ms(ctx, V, pot, l, r_c, E, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.log_derivatives(V, LEVELS, DELTA, RMAX, pot, l, r_c, E)
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if "logderiv_kernel" in e.name]
    if not ks:
        return None
    return float(np.median([e.device_time_total / 1e3 for e in ks]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, power, clock = card()
    with D.Context(0) as ctx:
        peak = ctx.measure_fp64_peak()
        res = ctx.solve_batch([D.Options(Z, LEVELS, RMAX, DELTA, 0.5, 0) for Z in range(1, 93)], keep_steps=False, radial=True)
        r = res[0].radial.r
        V = np.concatenate([x.radial.V for x in res])
        sass = loop_fp64_per_node()
        rec = dict(card=name, power_limit=power, max_sm_clock=clock, fp64_peak_tflops_measured=peak, sass=sass, cases={})
        setups = {
            "C3": (V, np.repeat(np.arange(92), 4), np.tile(np.arange(4), 92), 2.5, np.linspace(-2.0, 2.0, 1001)),
            "Ar": (V[17], 0, np.arange(4), 2.5, np.linspace(-2.0, 2.0, 301)),
        }
        for key, (v, pot, l, rc, E) in setups.items():
            out, t, ts = case(ctx, v, pot, l, rc, E, a.reps)
            steps = node_steps(out.r_c, r, len(E))
            km = kernel_ms(ctx, v, pot, l, rc, E, a.reps)
            c = dict(channels=int(out.D.shape[0]), energies=len(E), lanes=int(out.D.size), r_c_used=float(out.r_c[0]),
                     lane_node_steps=steps, call_ms_median=t * 1e3, call_ms_all=[x * 1e3 for x in ts],
                     kernel_ms_median=km if km is not None else "not measured",
                     lane_node_steps_per_s_call=steps / t,
                     all_finite=bool(np.isfinite(out.D).all()))
            if km:
                c["lane_node_steps_per_s_kernel"] = steps / (km * 1e-3)
                if sass and sass["fp64_per_node_step"]:
                    c["fp64_issue_share_of_measured_peak"] = steps * sass["fp64_per_node_step"] / (km * 1e-3) / (peak * 1e12 / 2)
            rec["cases"][key] = c
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
