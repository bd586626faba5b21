#!/usr/bin/env python
"""bench.py — atoms/sec of converged SCF on the periodic-table sweep (BASELINE.json metric), one process per GPU.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU solver on the host cores

A "step" is one pass of the hot path over one batch: the whole C3 workload (Z = 1..92, LDA, 14 multigrid levels =
16385 nodes, delta 0.0005, mixing 0.5, Rmax 25; SURVEY §8d) solved to the reference's stop criterion.  Weak scaling:
every rank solves one full sweep (atoms are independent, no collective on the data path), value = N*92 / max-rank time.
The strong-scaling figure (the same 92 atoms sharded over the ranks) is reported beside it under "strong_c3".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C3 = dict(levels=14, delta=0.0005, mixing=0.5, rmax=25.0, method=0)
WORKLOAD = "C3 periodic-table sweep Z=1-92 LDA, 14 levels (16385 nodes), delta 0.0005, mixing 0.5, Rmax 25"
STREAM_GROUPS_DEFAULT = 4          # libdftatom_b200's default (engine.cpp: stream_groups)
FLOP_PER_NODE_STEP = 11.0          # SURVEY §8(d) accounting convention for the Numerov shooting kernel
SEARCH_TRAFFIC_BYTES = 12553728    # DRAM bytes (read 12 551 424 + write 2 304) of one search_rows_kernel launch at full load, ncu --set full (profiles/r02_ncu_search_rows.txt)
REF_EXE = os.path.join(ROOT, "oracle", "_ref", "dftatom_ref")
ORACLE_EXE = os.path.join(ROOT, "oracle", "dftatom_oracle")


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Clocks and throttle reasons of the samples taken inside [t0, t1] (the timed region); the sampler is started before the
        warm-up steps so that nvidia-smi is already running, and if the timed region is too short to hold two samples the
        warm-up samples (same workload, same load) are used as well."""
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.12)
        self.proc.terminate()
        inside = [ln for ts, ln in self.lines if t0 is None or (t0 <= ts <= (t1 or ts) + 0.1)]
        window = "timed region"
        if len(inside) < 2:
            inside = [ln for ts, ln in self.lines]
            window = "warm-up + timed region"
        sm, smax, reasons = [], [], set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # under load = samples above the idle clock
        load = [x for x in sm if x > 0.5 * max(smax or [0])] or sm
        return dict(sm_mhz=statistics.median(load) if load else None, sm_max_mhz=max(smax) if smax else None,
                    reasons=sorted(reasons), samples=len(sm), window=window)


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm (also the cpu_baseline of the CUDA arm)
# ------------------------------------------------------------------------------------------------------------
def _golden_costs():
    """Per-Z single-core seconds of the unmodified reference on C3, recorded when tests/golden/sweep.json was made (used to order
    the pool longest-first and, only if the time budget runs out, to extrapolate the atoms that were not started)."""
    with open(os.path.join(ROOT, "tests", "golden", "sweep.json")) as f:
        g = json.load(f)
    return {a["options"]["Z"]: float(a["ref_seconds"]) for a in g["atoms"]}


def _cpu_exe():
    exe, kind = (REF_EXE, "reference") if os.path.exists(REF_EXE) else (ORACLE_EXE, "port")
    if not os.path.exists(exe):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "restatement"], check=True)
    return exe, kind


def _run_pool(exe, zs, cores, budget_s):
    """One single-threaded process of the reference's solver per atom (the solver is single-threaded), at most `cores` at a time,
    in the given order.  No new atom is started after budget_s.  Returns ({Z: seconds}, {Z: printed "Finished!"}, wall seconds)."""
    import tempfile
    t0 = time.time()
    pending = list(zs)
    running = {}
    secs, fin = {}, {}
    tmp = tempfile.mkdtemp(prefix="dftatom_ref_")
    while pending or running:
        while pending and len(running) < cores and time.time() - t0 < budget_s:
            z = pending.pop(0)
            out = open(os.path.join(tmp, f"{z}.txt"), "w")
            p = subprocess.Popen([exe, str(z), str(C3["levels"]), str(C3["mixing"]), str(C3["rmax"]), str(C3["delta"]), "0"], stdout=out)
            running[z] = (p, time.time(), out)
        if not running:
            break
        for z, (p, ts, out) in list(running.items()):
            if p.poll() is not None:
                secs[z] = time.time() - ts
                out.close()
                with open(out.name) as f:
                    fin[z] = "Finished!" in f.read()
                os.unlink(out.name)
                del running[z]
        time.sleep(0.005)
    try:
        os.rmdir(tmp)
    except OSError:
        pass
    return secs, fin, time.time() - t0


def cpu_reference_sweep(budget_s=420.0, cores=None, zs=None):
    """THE WHOLE C3 SWEEP (92 atoms) with the reference's own CPU solver (oracle/_ref/dftatom_ref = the unmodified reference compiled
    headless; falls back to the C restatement oracle/dftatom_oracle), P = all host cores, one process per atom, longest first
    (BASELINE.md section 3 / SURVEY 8d).  atoms/s = 92 / wall.  Only if budget_s runs out before every atom was started are the missing
    ones extrapolated from the recorded per-Z costs (flagged complete = False)."""
    cores = cores or os.cpu_count() or 1
    exe, kind = _cpu_exe()
    cost = _golden_costs()
    if zs:                                       # testing aid (--ref-atoms): a sub-list of the sweep
        cost = {z: cost[z] for z in zs}
    n_all = len(cost)
    order = sorted(cost, key=lambda z: -cost[z])
    secs, fin, wall = _run_pool(exe, order, cores, budget_s)
    done = sorted(secs)
    core_s = sum(secs.values())
    complete = len(done) == len(order)
    if complete:
        sweep_s = wall
        total_core_s = core_s
    else:
        ratio = core_s / sum(cost[z] for z in done)
        total_core_s = sum(cost.values()) * ratio
        sweep_s = max(total_core_s / cores, max(cost.values()) * ratio, wall)
    return dict(value=n_all / sweep_s, unit="atoms/s", cores=cores, kind=kind, complete=complete, atoms_run=len(done), atoms_finished=sum(fin.values()),
                wall_s=wall, core_seconds=core_s, sweep_core_seconds=total_core_s, per_core_atoms_per_s=n_all / total_core_s,
                sample=(f"the whole C3 sweep: {len(done)} of {n_all} atoms, one single-threaded process per atom on {cores} cores, longest first: "
                        f"{wall:.1f} s wall, {core_s:.0f} core-s, {sum(fin.values())} printed Finished!"
                        + ("" if complete else f"; time budget hit: the rest extrapolated from recorded per-Z costs => {total_core_s:.0f} core-s")))


def cpu_reference_sample(budget_s, cores=None):
    """A bounded, stratified sample of C3 for the CUDA arm's `cpu_baseline` key (10-30 s of CPU work): every 8th Z, one process per atom
    on all host cores; the sweep throughput is the LPT bound 92 / max(sum_cost/cores, max_cost) with every atom's recorded cost
    scaled by measured/recorded time of the sample.  (The reference arm, `--impl reference`, runs the whole sweep instead.)"""
    cores = cores or os.cpu_count() or 1
    exe, kind = _cpu_exe()
    cost = _golden_costs()
    cand = [z for z in range(4, 93, 8) if cost[z] <= budget_s] or [min(cost, key=cost.get)]
    sample = cand[:cores]
    secs, fin, wall = _run_pool(exe, sample, cores, 1e9)
    ratio = sum(secs.values()) / sum(cost[z] for z in sample)
    total = sum(cost.values()) * ratio
    longest = max(cost.values()) * ratio
    sweep_s = max(total / cores, longest)
    return dict(value=92.0 / sweep_s, unit="atoms/s", cores=cores, kind=kind,
                sample=f"Z={sample} of C3 run concurrently ({wall:.1f}s wall, {sum(secs.values()):.1f} core-s); per-Z costs of the full sweep "
                       f"scaled by {ratio:.3f} => {total:.0f} core-s, longest atom {longest:.1f}s; value = 92/max(core-s/cores, longest)",
                sweep_core_seconds=total, per_core_atoms_per_s=92.0 / total, wall_s=wall)


def run_reference_arm(a):
    """--impl reference: the reference's own CPU solver on the WHOLE configuration the CUDA arm runs (C3: 92 atoms), all host cores.
    The sweep is run ONCE, as one pool; its atoms are the arm's work, dealt over the --steps K "steps" (a step = 92 / K atoms' worth of
    the pool), so value = 92 / wall does not depend on K.  Warm-up: one hydrogen atom per core per warm-up step (pages the binary in)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    exe, kind = _cpu_exe()
    cores = os.cpu_count() or 1
    for _ in range(a.warmup):
        _run_pool(exe, [1] * min(cores, 4), cores, 1e9)
    r = cpu_reference_sweep(budget_s=a.ref_budget, zs=[int(z) for z in a.ref_atoms.split(",")] if a.ref_atoms else None)
    ms = r["wall_s"] * 1e3 / max(1, a.steps)
    v = r["value"]
    line = dict(impl="reference", metric="atoms/sec converged SCF (Z=1-92 LDA, 16385 nodes)", value=v, unit="atoms/s", n_gpus=a.gpus,
                steps=a.steps, warmup=a.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=dict(workload=WORKLOAD, atoms_converged=r["atoms_finished"],
                                              note="CPU: the whole 92-atom sweep as one pool of single-threaded reference processes on all host cores; "
                                                   "a step = its share of the pool (92 / steps atoms)"),
                cpu_baseline=dict(value=v, unit="atoms/s", cores=r["cores"], kind=r["kind"], sample=r["sample"], complete=r["complete"],
                                  core_seconds=r["core_seconds"], wall_s=r["wall_s"], atoms_finished=r["atoms_finished"]),
                e2e=dict(value=v, unit="atoms/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------------------
def run_cuda_arm(a):
    import torch
    import dftatom_b200 as D
    from dftatom_b200.shard import partition_atoms

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (dftatom_b200 has no CPU fallback)")
    # stdout carries exactly one JSON line: whatever libraries print on fd 1 meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    ctx = D.Context(local)
    opts = [D.Options(Z, C3["levels"], C3["rmax"], C3["delta"], C3["mixing"], C3["method"]) for Z in range(1, 93)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    def flush_l2():
        # the flush runs on torch's stream, the solve on the library's own (non-blocking) stream: order them explicitly
        flush.zero_()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        flush_l2()
        res = ctx.solve_batch(opts, keep_steps=False)

    dev_ms = 0.0
    launches = 0
    graph_iters = 0
    barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(a.steps):
        flush_l2()
        res = ctx.solve_batch(opts, keep_steps=False)      # host options in, host results out: the e2e path (production defaults)
        ms, nl = ctx.last_timing()
        h2d, d2h = ctx.last_transfer()                     # bytes this call copied (counted by the library from the buffers it copies)
        dev_ms += ms
        launches += nl
        graph_iters += ctx.last_graph_iterations()
    barrier()
    wall = time.perf_counter() - t0
    t_end = time.time()
    clocks = sampler.stop(t_end - wall, t_end) if rank == 0 else None
    if rank == 0 and a.dump_outputs:
        dump_outputs(res, a.dump_outputs)
    # Per-kernel-class CUDA-event timing (the roofline's kernel time): the production path replays the SCF loop from ONE CUDA-graph launch
    # (while node, device-side condition), where host-side events cannot be recorded between the kernels; so the same sweep is run
    # `steps` more times, back to back with the timed ones, with set_option("profile", 1) - the host-driven loop with an event pair around
    # every kernel class.  Identical kernels, identical records (tests); its device time is reported beside the timed one.
    prof = {k: dict(ms=0.0, launches=0, work=0.0) for k in D.api.KERNEL_CLASSES}
    prof_dev_ms = 0.0
    ctx.set_option("profile", 1)
    ctx.set_option("stream_groups", 1)      # one chain: the class times add up to the sweep (the production default overlaps 4 groups of atoms on 4 streams)
    for _ in range(a.steps):
        flush_l2()
        ctx.solve_batch(opts, keep_steps=False)
        prof_dev_ms += ctx.last_timing()[0]
        for k, v in ctx.last_profile().items():
            for f in ("ms", "launches", "work"):
                prof[k][f] += v[f]
    # the same kernel at full load: the first 24 SCF steps of the sweep, where all 92 atoms (916 orbitals) are still active - the whole-sweep figure
    # above averages in the 70-step tail in which 3-10 atoms keep 148 SMs busy
    full_load = None
    if rank == 0:
        ctx.set_option("step_cap", 24)
        flush_l2()
        ctx.solve_batch(opts, keep_steps=False)
        pf = ctx.last_profile()["search"]
        full_load = dict(scf_steps=24, lane_node_steps=pf["work"], kernel_ms=pf["ms"])
        ctx.set_option("step_cap", 0)
    ctx.set_option("profile", 0)
    ctx.set_option("stream_groups", STREAM_GROUPS_DEFAULT)

    wall = max_over_ranks(wall)
    dev_s = max_over_ranks(dev_ms * 1e-3)
    n_atoms_total = len(opts) * world * a.steps
    n_finished = int(sum_over_ranks(sum(r.finished for r in res)))
    n_capped = len(opts) - sum(r.finished for r in res)

    # strong scaling on C3 as given: the same 92 atoms sharded over the ranks (LPT by orbital count)
    strong = None
    if world > 1:
        mine = partition_atoms([o.Z for o in opts], world)[rank]
        my_opts = [opts[i] for i in mine]
        ctx.solve_batch(my_opts, keep_steps=False)
        tws, tds = [], []
        for _ in range(3):
            barrier()
            t1 = time.perf_counter()
            r_mine = ctx.solve_batch(my_opts, keep_steps=False)
            barrier()
            tws.append(max_over_ranks(time.perf_counter() - t1))
            tds.append(max_over_ranks(ctx.last_timing()[0] * 1e-3))
        tw, td = min(tws), min(tds)
        ctx.set_option("profile", 1); ctx.set_option("stream_groups", 1)
        ctx.solve_batch(my_opts, keep_steps=False)
        ctx.set_option("profile", 0); ctx.set_option("stream_groups", STREAM_GROUPS_DEFAULT)
        pr_s = ctx.last_profile()
        tot = sum(v["ms"] for v in pr_s.values()) or 1.0
        longest = max(r.n_steps for r in r_mine) if r_mine else 0
        longest = int(max_over_ranks(longest))
        strong = dict(value=92.0 / tw, value_device=92.0 / td, unit="atoms/s", scaling="strong", atoms=92, seconds=tw, device_seconds=td,
                      efficiency_vs_1gpu=None, longest_chain_steps=longest, ms_per_step_of_longest_chain=td * 1e3 / max(1, longest),
                      limiting_kernel=max(pr_s, key=lambda k_: pr_s[k_]["ms"]), kernel_share_rank0={k_: v["ms"] / tot for k_, v in pr_s.items()},
                      note="the same 92 atoms sharded over the ranks (dftatom_partition: LPT on orbitals x expected SCF steps); bounded below by the "
                           "dependent chain of the slowest atom (Z=68-70: 100 SCF steps), not by throughput")

    if rank == 0:
        peak = ctx.measure_fp64_peak()
        s = prof["search"]
        achieved = FLOP_PER_NODE_STEP * s["work"] / (s["ms"] * 1e-3) / 1e12 if s["ms"] > 0 else 0.0
        shares = {k: (v["ms"] / (prof_dev_ms or 1.0)) for k, v in prof.items()}
        if full_load and full_load["kernel_ms"] > 0:
            full_load["achieved"] = FLOP_PER_NODE_STEP * full_load["lane_node_steps"] / (full_load["kernel_ms"] * 1e-3) / 1e12
            full_load["frac"] = full_load["achieved"] / peak if peak else None
            full_load["note"] = ("same kernel, same convention, restricted to SCF steps 0-23 of the sweep (all 92 atoms active); the headline frac is the whole "
                                 "sweep including the tail where 3-10 atoms remain")
        line = dict(
            metric="atoms/sec converged SCF (Z=1-92 LDA, 16385 nodes)", value=n_atoms_total / dev_s, unit="atoms/s", n_gpus=world,
            steps=a.steps, warmup=a.warmup, ms_per_step=wall * 1e3 / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="f64", data="synthetic",
            config=dict(workload=WORKLOAD, atoms_per_gpu=92, l2="flushed between steps (256 MiB memset, synchronised before the solve)",
                        atoms_converged=n_finished,
                        note=f"every rank solves one full sweep; on rank 0 {len(opts) - n_capped}/92 atoms met the reference's stop test and {n_capped} ran to the "
                             "100-step cap (the reference: 89 / 3, Z=68-70); `value` counts all 92 like the reference's sweep does"),
            e2e=dict(value=n_atoms_total / wall, unit="atoms/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                     note="options (host structs) in, per-atom results (host structs) out through dftatom_solve_batch; the bytes are what the library "
                          "copied for one sweep (atom / orbital descriptors up; per-atom state + last step record down); grid tables are cached per context"),
            gpu_launches=int(launches),
            scf_loop=dict(mode="CUDA-graph while node, loop condition set on the device (cudaGraphSetConditional)" if graph_iters else "host-driven loop",
                          scf_steps_inside_graph=int(graph_iters), device_ms_per_sweep=dev_ms / a.steps,
                          device_ms_per_sweep_profiled_host_loop=prof_dev_ms / a.steps, stream_groups=STREAM_GROUPS_DEFAULT,
                          note="timed sweeps: the library's defaults - the 92 atoms dealt into 4 groups whose SCF chains run concurrently on 4 streams, each group's loop "
                               "one CUDA-graph launch; profiled sweeps: one group, host-driven loop, CUDA events around every kernel class"),
            roofline=dict(kernel="search_rows_kernel (Numerov shooting: Sturm-count search; one CTA per orbital, lane = radial segment (128 per orbital), every thread "
                                 "4 trial energies x 2 basis chains: 11 FP64 instructions per credited (trial energy, node) = 11 FLOP -> ceiling 0.5 of the FMA peak)",
                          bound="fp64", achieved=achieved, peak=peak, unit="TFLOP/s",
                          frac=achieved / peak if peak else None, traffic=SEARCH_TRAFFIC_BYTES,
                          traffic_source="dram__bytes_read + write of one search_rows_kernel launch with all 916 orbitals active, ncu --set full "
                                         "(profiles/r02_ncu_search_rows.txt): the kernel is FP64-bound, its tables stay in L2",
                          peak_source="measured live: DFMA microbench in libdftatom_b200 (MEASURED_PEAKS.json has no FP64 entry)",
                          flop_per_lane_node_step=FLOP_PER_NODE_STEP, lane_node_steps=s["work"], kernel_ms=s["ms"], share_of_step=shares, full_load=full_load,
                          timing="CUDA events around every kernel class over `steps` profiled sweeps run back to back with the timed ones (see scf_loop)"),
            kernels={k: dict(ms=v["ms"], launches=int(v["launches"]), work=v["work"]) for k, v in prof.items()},
            search=dict(orbital_solves=prof["match"]["work"], rounds_per_solve=prof["density"]["work"] / max(1.0, prof["match"]["work"]),
                        inward_sweeps_per_solve_reference=140, note="one round = 4 concurrent inward sweeps (trial energies), 128 radial segments each"),
            poisson=dict(poisson_record(prof, len(opts), a.steps), share_of_step=shares["poisson"]),
            clocks=clocks,
        )
        if strong:
            strong["efficiency_vs_1gpu"] = None     # the driver computes efficiencies from the per-N lines; 1-GPU value of the same metric = this line at N=1
            line["strong_c3"] = strong
            line["value_strong"] = strong["value"]
            line["scaling_strong"] = "strong: the same 92 atoms sharded over the ranks (see strong_c3)"
        # The legs below are extras beside the headline line: a failure in one of them (e.g. the 50 GiB of the C5a leg not being
        # available) is recorded under its key and must not cost the line itself.
        def leg(key, fn):
            try:
                line[key] = fn()
            except Exception as e:          # noqa: BLE001
                line[key] = dict(error=f"{type(e).__name__}: {e}")
                torch.cuda.empty_cache()

        def leg_batch():
            # the same sweep replicated 8x in ONE batch (736 atoms): C3 as given is bounded by the SCF chain of its slowest atoms
            # (from step ~35 on fewer than 30 atoms are left), a larger batch shows what the kernels sustain when the GPU is full
            big = opts * 8
            ctx.solve_batch(big, keep_steps=False)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            ctx.solve_batch(big, keep_steps=False)
            tb = time.perf_counter() - t1
            dev_b = ctx.last_timing()[0]
            ctx.set_option("profile", 1); ctx.set_option("stream_groups", 1)
            ctx.solve_batch(big, keep_steps=False)
            ctx.set_option("profile", 0); ctx.set_option("stream_groups", STREAM_GROUPS_DEFAULT)
            prb = ctx.last_profile()
            sb_ = prb["search"]
            ach = FLOP_PER_NODE_STEP * sb_["work"] / (sb_["ms"] * 1e-3) / 1e12 if sb_["ms"] > 0 else 0.0
            return dict(value=len(big) / tb, unit="atoms/s", atoms=len(big), seconds=tb, device_ms=dev_b,
                        search_roofline=dict(bound="fp64", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak if peak else None, kernel_ms=sb_["ms"],
                                             lane_node_steps=sb_["work"], note="the energy search with 7328 orbitals in flight (search_rows_kernel: one CTA per orbital)"),
                        kernels={k_: round(v["ms"], 2) for k_, v in prb.items()},
                        note="8 copies of the Z=1-92 sweep in one dftatom_solve_batch call, host options in, host results out")

        def leg_rn():
            # second half of BASELINE.json's metric: wall-ms of one Radon SCF (C2: Z=86 LSDA, 17 levels = 131073 nodes, delta 1e-4,
            # mixing 0.5, Rmax 50) through the same public call, host options in, host results out; warm-up run first
            rn = [D.Options(86, 17, 50.0, 0.0001, 0.5, 1)]
            ctx.solve_batch(rn, keep_steps=False)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            r_rn = ctx.solve_batch(rn, keep_steps=False)[0]
            rn_ms = (time.perf_counter() - t1) * 1e3
            return dict(metric="Rn SCF ms", value=rn_ms, unit="ms", device_ms=ctx.last_timing()[0], scf_steps=r_rn.n_steps, finished=bool(r_rn.finished),
                        Etotal=r_rn.Etotal, workload="C2 Radon Z=86 LSDA, 17 levels (131073 nodes), delta 0.0001, mixing 0.5, Rmax 50",
                        reference_cpu_seconds_1core=518.0, reference_source="SURVEY.md section 6 (unmodified reference, g++ -O2, one core)")

        def leg_cpu():
            cb = cpu_reference_sample(30.0)
            return {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}

        def leg_c1():
            # BASELINE configs[0]: Argon through the same public call
            ar = [D.Options(18, C3["levels"], C3["rmax"], C3["delta"], C3["mixing"], 0)]
            ctx.solve_batch(ar, keep_steps=False)
            t1 = time.perf_counter()
            r_ar = ctx.solve_batch(ar, keep_steps=False)[0]
            w_ms = (time.perf_counter() - t1) * 1e3
            return dict(metric="Ar SCF ms", value=w_ms, unit="ms", device_ms=ctx.last_timing()[0], scf_steps=r_ar.n_steps, finished=bool(r_ar.finished), Etotal=r_ar.Etotal,
                        workload="C1 Argon Z=18 LDA, 14 levels (16385 nodes), delta 0.0005, mixing 0.5, Rmax 25")

        def leg_c4():
            # BASELINE configs[3]: the 25-atom LSDA open-shell batch at 65537 nodes
            zs = list(range(21, 31)) + list(range(57, 72))
            c4 = [D.Options(z, 16, 50.0, 0.0002, 0.5, 1) for z in zs]
            ctx.solve_batch(c4, keep_steps=False)
            t1 = time.perf_counter()
            r4 = ctx.solve_batch(c4, keep_steps=False)
            w_ms = (time.perf_counter() - t1) * 1e3
            dev4 = ctx.last_timing()[0]
            ctx.set_option("profile", 1); ctx.set_option("stream_groups", 1)
            ctx.solve_batch(c4, keep_steps=False)
            ctx.set_option("profile", 0); ctx.set_option("stream_groups", STREAM_GROUPS_DEFAULT)
            pr4 = ctx.last_profile()
            return dict(metric="C4 batch ms", value=w_ms, unit="ms", device_ms=dev4, atoms=len(c4), atoms_per_s=len(c4) / (w_ms * 1e-3),
                        atoms_converged=sum(r.finished for r in r4), kernels={k_: round(v["ms"], 2) for k_, v in pr4.items()},
                        workload="C4 LSDA open-shell batch Z=21-30,57-71, 16 levels (65537 nodes), delta 0.0002, mixing 0.5, Rmax 50",
                        reference_cpu_core_seconds=8922.0, reference_source="SURVEY.md B.4 (unmodified reference, g++ -O2, sum over the 25 atoms)")

        if world == 1 and not a.no_batch:
            leg("batch_8xC3", leg_batch)
            leg("c1_argon", leg_c1)
            leg("c4_lsda_batch", leg_c4)
        def leg_damping():
            # SURVEY 8(f) rank 4, opt-in (beyond the reference): per-atom damping raised when Etotal sloshes with period 2
            ctx.set_option("adaptive_mixing", 1)
            try:
                ctx.solve_batch(opts, keep_steps=False)
                t1 = time.perf_counter()
                rd = ctx.solve_batch(opts, keep_steps=False)
                wd = time.perf_counter() - t1
            finally:
                ctx.set_option("adaptive_mixing", 0)
            return dict(value=len(opts) / wd, unit="atoms/s", atoms_converged=sum(r.finished for r in rd), scf_steps=sum(r.n_steps for r in rd),
                        scf_steps_default=sum(r.n_steps for r in res), atoms_converged_default=sum(r.finished for r in res), device_ms=ctx.last_timing()[0],
                        note="set_option('adaptive_mixing', 1): NOT the reference's algorithm (default off); Er, Tm, Yb converge instead of running 100 steps")

        if world == 1 and not a.no_batch:
            leg("c3_adaptive_mixing_opt_in", leg_damping)
        if world == 1 and not a.no_parity:
            leg("parity", lambda: parity_block(ctx, D))
        if world == 1 and not a.no_rn:
            leg("rn_scf", leg_rn)
        if world == 1 and not a.no_micro:
            # BASELINE.json configs[4]: the two kernels at scale, each against its own roofline
            leg("c5b_numerov_lanes", lambda: micro_c5b(ctx, peak, cpu_baseline=not a.no_cpu_baseline))
            leg("c5a_poisson_vcycle", lambda: micro_c5a(ctx, torch, _hbm_peak(), n_dens=a.micro_densities, cpu_baseline=not a.no_cpu_baseline))
        if world == 1 and not a.no_cpu_baseline:
            leg("cpu_baseline", leg_cpu)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(res, out_dir):
    """What the last timed sweep returned to its caller, atoms in input order (Z = 1..92), one float64 array per DIR/<name>.npy:
    energies [atom][Etotal, Ekin, Ecoul, Eenuc, Exc]; n_steps [atom]; status [atom] (0 = converged); n_levels [atom][spin] (0 for the
    second spin of an unpolarised atom).  The levels of all atoms are concatenated in (atom, spin) order, n_levels of them per block:
    eigenvalues [level] and levels [level][n, l, occ, nodes] in (n, l) order, sorted_levels [level][n, l, occ, nodes, E] in eigenvalue
    order.  A result with a non-finite value is an error: nothing is written and ValueError names the atoms."""
    import numpy as np
    n_levels = np.zeros((len(res), 2), np.float64)
    eig, levels, sorted_levels = [], [], []
    for i, r in enumerate(res):
        for s, (chan, schan) in enumerate(zip(r.levels, r.sorted_levels)):
            n_levels[i, s] = len(chan)
            eig += [L.E for L in chan]
            levels += [(L.n, L.l, L.occ, L.nodes) for L in chan]
            sorted_levels += [(L.n, L.l, L.occ, L.nodes, L.E) for L in schan]
    arrays = dict(energies=np.array([[r.Etotal, r.Ekin, r.Ecoul, r.Eenuc, r.Exc] for r in res], np.float64),
                  n_steps=np.array([r.n_steps for r in res], np.float64), status=np.array([r.status for r in res], np.float64),
                  n_levels=n_levels, eigenvalues=np.array(eig, np.float64), levels=np.array(levels, np.float64).reshape(-1, 4),
                  sorted_levels=np.array(sorted_levels, np.float64).reshape(-1, 5))
    bad = sorted({r.options.Z for r in res if not np.isfinite([r.Etotal, r.Ekin, r.Ecoul, r.Eenuc, r.Exc]
                                                             + [L.E for ch in r.levels + r.sorted_levels for L in ch]).all()})
    if bad:
        raise ValueError(f"--dump-outputs: non-finite energies or eigenvalues in the results of Z = {bad}")
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), x)


def poisson_record(prof, n_atoms, steps):
    """The other half of the C3 step: the Poisson solves (SURVEY 8d row 3: grid on chip at 16385 nodes - not an HBM kernel).  Live numbers:
    CUDA-event time of the class, Gauss-Seidel node updates counted by the kernels, V-cycle equivalents (12 N updates each).  The shared-memory
    bandwidth and pipe utilisation come from the ncu capture of the same kernel (profiles/)."""
    p = prof["poisson"]
    N = (1 << C3["levels"]) + 1
    ups = p["work"] / (p["ms"] * 1e-3) if p["ms"] else None
    return dict(kernel="poisson_direct_kernel (warm solves in increment form from SCF step 4 on: the increment's level-0 tridiagonal system solved directly - "
                       "Thomas algorithm as block scans of affine maps, one CTA per density) + poisson_warm_kernel (SCF steps 1-3: 7 V-cycles on the increment, "
                       "one CTA per density, level visits in registers) + poisson_full_kernel (cold full-multigrid solves of the initial guess and SCF step 0)",
                launches=int(p["launches"]), node_updates=p["work"], ms=p["ms"], node_updates_per_s=ups,
                share_of_step=None,
                bound="latency: a direct solve is ~12 k cycles on one SM per density (two scans over the grid, 40 N bytes of L2 / HBM traffic), a V-cycle solve "
                      "~250 dependent Gauss-Seidel sweeps; neither comes near a bandwidth or FLOP limit on this grid (16385 nodes: the whole hierarchy is on chip)",
                note="node_updates = Gauss-Seidel node updates of the V-cycle solves + 2 N per direct solve (its two elimination passes)",
                ncu="profiles/r02_ncu_poisson_direct.txt, profiles/r02_ncu_poisson_warm.txt, profiles/r02_ncu_poisson_cluster.txt")


def parity_block(ctx, D):
    """Worst deviation of the PRODUCTION path from the committed goldens of the unmodified reference (tests/golden/*.json), per config, over
    every SCF step both ran: eigenvalues (north_star: 1e-6 Ha) and the five energies (1e-5 Ha).  `reference_self` = how far the reference
    lands from ITSELF when mixing changes by one unit in the last place (tests/golden/self_repro.json), for the atoms that have such a run."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    keys = ("Etotal", "Ekin", "Ecoul", "Eenuc", "Exc")
    out = {}

    def load(name):
        with open(os.path.join(ROOT, "tests", "golden", name + ".json")) as f:
            return json.load(f)["atoms"]

    def tables(at):
        n_ref = at.get("n_steps", len(at["steps"]))
        if "energies_per_step" in at:
            return n_ref, at["eig_per_step"], at["energies_per_step"]
        return n_ref, [[l["E"] for l in s["levels"]] for s in at["steps"]], [[s[k] for k in keys] for s in at["steps"]]

    try:
        selfr = load("self_repro")
    except OSError:
        selfr = []
    for name, label in (("argon", "C1"), ("sweep", "C3"), ("radon", "C2"), ("lsda_batch", "C4")):
        atoms = load(name)
        res = ctx.solve_batch([D.Options(t["options"]["Z"], t["options"]["levels"], t["options"]["rmax"], t["options"]["delta"], t["options"]["mixing"],
                                         t["options"]["method"]) for t in atoms])
        de = dE = 0.0
        worst = None
        same_stop = 0
        for r, at in zip(res, atoms):
            n_ref, eigs, en = tables(at)
            n = min(r.n_steps, n_ref)
            same_stop += int(r.n_steps == n_ref)
            for k in range(n):
                st = r.steps[k]
                de = max(de, float(np.max(np.abs(np.array([x for ch in st.E for x in ch]) - np.array(eigs[k])))))
                d5 = max(abs(getattr(st, key) - en[k][j]) for j, key in enumerate(keys))
                if d5 > dE:
                    dE, worst = d5, (at["options"]["Z"], k)
        rec = dict(atoms=len(atoms), max_abs_eig_dev_Ha=de, max_abs_energy_dev_Ha=dE, worst_energy_at=dict(Z=worst[0], step=worst[1]) if worst else None,
                   same_stop_step=same_stop, atoms_finished=sum(r.finished for r in res), reference_finished=sum(bool(t["finished"]) for t in atoms),
                   north_star=dict(eig=1e-6, energy=1e-5))
        noise = 0.0
        for sr in selfr:
            for at in atoms:
                if at["options"]["Z"] == sr["options"]["Z"] and at["options"]["levels"] == sr["options"]["levels"] and at["options"]["method"] == sr["options"]["method"]:
                    n_ref, eigs, en = tables(at)
                    n = min(n_ref, sr["n_steps"])
                    noise = max(noise, max(abs(sr["energies_per_step"][k][j] - en[k][j]) for k in range(n) for j in range(5)))
        if noise:
            rec["reference_self_max_abs_energy_dev_Ha"] = noise
        out[label] = rec
    out["note"] = ("production path (8 V-cycles, FMA, warm start) vs tests/golden; the -m gpu tests assert C1/C3 at north_star outright and C2/C4 in the "
                   "bit-reproducible Poisson mode (set_option poisson_exact), where the only excess over 1e-5 Ha is on atoms the reference does not reproduce itself")
    return out


# ------------------------------------------------------------------------------------------------------------
# kernel micro-benchmarks (BASELINE.json configs[4], SURVEY 8d: C5a Poisson V-cycle, C5b Numerov lanes)
# ------------------------------------------------------------------------------------------------------------
def _splitmix64_unit(seed, n):
    """k-th output of splitmix64(seed) / 2^64, k = 0..n-1 (SURVEY 8d, C5a)."""
    import numpy as np
    out = np.empty(n, np.float64)
    x = seed & 0xFFFFFFFFFFFFFFFF
    M = 0xFFFFFFFFFFFFFFFF
    for k in range(n):
        x = (x + 0x9E3779B97F4A7C15) & M
        z = x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        z = z ^ (z >> 31)
        out[k] = z / 2.0 ** 64
    return out


def micro_c5a(ctx, torch, hbm_peak_gbs, n_dens=1024, levels=20, delta=1.25e-5, rmax=50.0, cycles=8, reps=3, cpu_baseline=True):
    """C5a: batched Poisson V-cycle on 2^20+1 nodes x 1024 densities rho_k = Z_k a_k^3/pi exp(-2 a_k r) (SURVEY 8d), boundary
    values (0, Z_k), device-resident.  Unit of work = one reference-shaped V-cycle on all densities; algorithmic traffic
    112 B x N per V-cycle per density."""
    import numpy as np
    N = (1 << levels) + 1
    ld = N + 3
    Zk = 1.0 + (np.arange(n_dens) % 92)
    ak = 0.5 + 3.5 * _splitmix64_unit(20261017, n_dens)
    dev = torch.device("cuda")
    i = torch.arange(N, dtype=torch.float64, device=dev)
    rp = rmax / (np.exp((N - 1) * delta) - 1.0)
    ex = torch.exp(i * delta)
    r = rp * (ex - 1.0)
    psrc = r * (4.0 * np.pi * rp * rp * delta * delta) * ex * ex           # r 4 pi K_i, K_i = Rp^2 delta^2 e^{2 delta i}
    psrc[0] = 0.0; psrc[-1] = 0.0
    d_src = torch.zeros((n_dens, ld), dtype=torch.float64, device=dev)
    d_phi = torch.zeros((n_dens, ld), dtype=torch.float64, device=dev)
    tZ = torch.from_numpy(Zk).to(dev); ta = torch.from_numpy(ak).to(dev)
    for k0 in range(0, n_dens, 32):
        k1 = min(k0 + 32, n_dens)
        a_ = ta[k0:k1, None]
        d_src[k0:k1, :N] = psrc[None, :] * (tZ[k0:k1, None] * a_ ** 3 / np.pi) * torch.exp(-2.0 * a_ * r[None, :])
    sb = ctx.poisson_scratch_bytes(levels, n_dens)
    scratch = torch.empty(sb // 8, dtype=torch.float64, device=dev)

    def reset():
        d_phi.zero_()
        d_phi[:, N - 1] = tZ
        torch.cuda.synchronize()

    out = dict(workload=f"C5a Poisson V-cycle, {N} nodes x {n_dens} densities, delta {delta}, Rmax {rmax}, device-resident "
                        f"({(2 * n_dens * ld * 8 + sb) / 2 ** 30:.1f} GiB >> L2)",
               bytes_per_vcycle_algorithmic=112.0 * N * n_dens)
    best = {}
    for name, ncyc, fuse in (("single", 1, False), ("chained", cycles, True)):
        times = []
        for rep in range(reps + 1):                  # first repetition = warm-up
            reset()
            ms, nl = ctx.poisson_vcycles_dev(levels, delta, n_dens, d_phi.data_ptr(), d_src.data_ptr(), ld, scratch.data_ptr(), sb, ncyc, fuse)
            if rep:
                times.append(ms / ncyc)
        best[name] = dict(ms_per_vcycle=statistics.median(times), launches_per_call=nl, vcycles_per_call=ncyc)
    for name, b in best.items():
        b["vcycles_per_s"] = n_dens / (b["ms_per_vcycle"] * 1e-3)
        b["achieved_gbs"] = 112.0 * N * n_dens / (b["ms_per_vcycle"] * 1e-3) / 1e9
        b["frac_of_hbm_peak"] = b["achieved_gbs"] / hbm_peak_gbs
    out["single_vcycle"] = best["single"]
    out["chained_vcycles"] = best["chained"]
    out["chained_vcycles"]["note"] = (f"{cycles} V-cycles per call; the last visit of level 0 of one cycle and the first of the next are one "
                                      "pass (6 sweeps): actual level-0 traffic 56+28 B/node instead of 2 x 56")
    # known answer: after `cycles` V-cycles from zero, U_k -> Z_k (1 - exp(-2 a_k r)(1 + a_k r)) up to the discretisation error
    ks = [0, n_dens // 2, n_dens - 1]
    err = 0.0
    for k in ks:
        ux = Zk[k] * (1.0 - torch.exp(-2.0 * ak[k] * r) * (1.0 + ak[k] * r))
        err = max(err, float(torch.max(torch.abs(d_phi[k, :N] - ux))) / Zk[k])
    out["known_answer_max_err_over_Z"] = err
    # roofline of the leg = ONE reference-shaped V-cycle (every level read and written once per leg: the 112 B/node are really
    # moved); the chained figure credits 112 B/node while its fused tops move 84 on level 0, so it can exceed the copy peak
    out["roofline"] = dict(kernel="stream_visit_kernel (+ poisson_mid_kernel for the levels of <= 2048 nodes)", bound="hbm",
                           achieved=best["single"]["achieved_gbs"], peak=hbm_peak_gbs, unit="GB/s",
                           frac=best["single"]["achieved_gbs"] / hbm_peak_gbs, traffic=27.2 * N * n_dens,
                           traffic_source="ncu --set full of the level-0 down-visit (profiles/r01_ncu_stream_visit.txt): dram read 16.0 + write 11.2 "
                                          "B/node against the algorithmic 16 + 12 of that launch; scaled here to this launch's nodes x densities",
                           bytes_per_node_per_vcycle=112.0, peak_source="MEASURED_PEAKS.json hbm copy (fallback 6459 GB/s)")
    if cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        k = n_dens - 1
        src_h = d_src[k, :N].cpu().numpy(); phi_h = np.zeros(N); phi_h[-1] = Zk[k]
        t0 = time.time()
        o, _ = O.poisson_vcycles(levels, delta, phi_h, src_h, cycles)
        dt = time.time() - t0
        out["cpu_baseline"] = dict(value=cycles / dt, unit="V-cycles/s (one density)", cores=1, kind="port",
                                   sample=f"{cycles} V-cycles of density {k} with the oracle's PoissonSolver restatement ({dt:.2f} s)",
                                   max_abs_diff_gpu_vs_oracle=float(np.max(np.abs(d_phi[k, :N].cpu().numpy() - o))))
    del d_src, d_phi, scratch
    torch.cuda.empty_cache()
    return out


def micro_c5b(ctx, fp64_peak_tflops, reps=20, cpu_baseline=True):
    """C5b: 4096 lanes = 16 (n,l) x 256 trial energies in [1.5 E_n, 0.5 E_n], E_n = -Z^2/2n^2, V = -Z/r, Z = 86, on C2's grid
    (131073 nodes, delta 1e-4, Rmax 50); each lane = one inward sweep returning (sign y0, node count)."""
    import numpy as np
    levels, delta, rmax, Z = 17, 1e-4, 50.0, 86
    N = (1 << levels) + 1
    rp = rmax / (np.exp((N - 1) * delta) - 1.0)
    r = rp * (np.exp(np.arange(N) * delta) - 1.0)
    V = np.zeros(N); V[1:] = -Z / r[1:]
    shells = [(1, 0), (2, 0), (2, 1), (3, 0), (3, 1), (3, 2), (4, 0), (4, 1), (4, 2), (4, 3), (5, 0), (5, 1), (5, 2), (5, 3), (6, 0), (6, 1)]
    ls, Es = [], []
    for n, l in shells:
        En = -Z * Z / (2.0 * n * n)
        Es.append(np.linspace(1.5 * En, 0.5 * En, 256)); ls.append(np.full(256, l, np.int32))
    Es = np.concatenate(Es); ls = np.concatenate(ls); lim = np.zeros(len(Es), np.int32)
    # two shapes of the same sweep: serial in r (one warp = 32 energies walks the whole grid) and parallel in r (one cluster
    # of 4 CTAs per 32 energies, warp = one of 16 radial segments; the Sturm count comes from the segments' transfer matrices alone)
    kernels = {}
    # rows (production search sweep): lanes across the radial grid, 4 / 16 energies per CTA on 128 / 32 segments
    for name, impl in (("serial_in_r", 0), ("parallel_in_r", 2), ("rows_4x128", 4), ("rows_16x32", 6)):
        ctx.set_option("r_segments", 16 if impl == 2 else -1)          # 16 segments (clusters of 4 CTAs) measured best for these lanes
        try:
            sign, lg, cnt, ms, steps = ctx.numerov_lanes_timed(V, levels, delta, rmax, ls, Es, lim, impl=impl, reps=reps)
        finally:
            ctx.set_option("r_segments", -1)
        # known answer: the Sturm count of a lane = number of Coulomb levels n' > l with -Z^2/2n'^2 below its energy (+1
        # throughout for l = 3, SURVEY fact 6); it steps from n-l-1 to n-l where E crosses E_n
        ok = True
        for g, (n, l) in enumerate(shells):
            e = Es[g * 256:(g + 1) * 256]
            want = sum((-Z * Z / (2.0 * q * q) < e).astype(np.int64) for q in range(l + 1, 40))
            ok = ok and bool((cnt[g * 256:(g + 1) * 256] - (1 if l == 3 else 0) == want).all())
            ok = ok and int(want[127]) == n - l - 1 and int(want[128]) == n - l
        tf = 11.0 * steps / (ms * 1e-3) / 1e12
        kernels[name] = dict(ms_per_launch=ms, lanes_per_s=len(Es) / (ms * 1e-3), achieved_tflops=tf, known_answer_ok=ok)
    best = max(kernels, key=lambda k_: kernels[k_]["achieved_tflops"])
    tf = kernels[best]["achieved_tflops"]
    out = dict(workload="C5b Numerov shooting, 4096 (orbital, trial-energy) lanes, Z=86 Coulomb well, 131073 nodes",
               lane_node_steps=steps, kernels=kernels, known_answer_ok=all(k_["known_answer_ok"] for k_ in kernels.values()),
               roofline=dict(kernel={"serial_in_r": "numerov_lanes_fast_kernel", "parallel_in_r": "numerov_lanes_seg_kernel", "rows_4x128": "numerov_lanes_rows_kernel",
                                     "rows_16x32": "numerov_lanes_rows_kernel"}[best] + f" ({best})",
                             bound="fp64", achieved=tf, peak=fp64_peak_tflops, unit="TFLOP/s",
                             frac=tf / fp64_peak_tflops if fp64_peak_tflops else None, traffic=None, flop_per_lane_node_step=11.0,
                             note="credited 11 FLOP per (lane, node-step) whatever the kernel executes (SURVEY 8d); 4096 lanes are 128 warps "
                                  "for 148 SMs x 4 FP64 pipes, so the serial sweep cannot fill the machine; the parallel-in-r and rows kernels execute 11 FP64 "
                                  "instructions per (lane, node) for the two basis chains of a segment's transfer matrix: their ceiling is 0.5 of the FMA peak"))
    if cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        sel = np.arange(0, len(Es), 16)
        t0 = time.time()
        O.numerov_lanes(V, delta, rmax, ls[sel], Es[sel], lim[sel])
        dt = time.time() - t0
        out["cpu_baseline"] = dict(value=len(sel) / dt, unit="lanes/s", cores=1, kind="port",
                                   sample=f"every 16th lane ({len(sel)} lanes) with the oracle's CountNodes + SolutionInZero restatement ({dt:.2f} s)")
    return out


def _hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        for key in ("hbm_gbs", "hbm_copy_gbs", "hbm_GBps", "hbm"):
            if key in m:
                v = m[key]
                return float(v["burst"] if isinstance(v, dict) and "burst" in v else (v["value"] if isinstance(v, dict) else v))
    except Exception:
        pass
    return 6459.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-budget", type=float, default=420.0, help="--impl reference: seconds after which no further atom of the sweep is started")
    ap.add_argument("--ref-atoms", default="", help="--impl reference, testing aid: comma list of Z to run instead of the whole sweep")
    ap.add_argument("--no-rn", action="store_true", help="skip the Radon (C2) SCF timing")
    ap.add_argument("--no-batch", action="store_true", help="skip the replicated-batch (8 x C3) throughput figure and the C1 / C4 timings")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity block (worst deviation from the committed reference goldens per config)")
    ap.add_argument("--no-micro", action="store_true", help="skip the kernel micro-benchmarks (C5a Poisson V-cycle, C5b Numerov lanes)")
    ap.add_argument("--micro-densities", type=int, default=1024, help="densities of the C5a micro-benchmark (1024 = BASELINE.json; ~34 GiB)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one returned (per-atom energies, eigenvalues, level tables) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs records the CUDA arm's results; the reference arm has none to write")
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_cuda_arm(a)


if __name__ == "__main__":
    main()
