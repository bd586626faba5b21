"""Round-2 kernels under compute-sanitizer (memcheck / racecheck): the rows search (numerov_rows.cu: all three round shapes, lanes entry), the
one-CTA warm Poisson kernel (poisson_warm.cu) with the exact coarse solve, the direct warm Poisson solve (poisson_direct.cu).  Small grids and
a low step cap: the tools slow the kernels down 20-100x."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import dftatom_b200 as D
ctx = D.Context(0)
ctx.set_option("use_graph", int(os.environ.get("SAN_GRAPH", "0")))
ctx.set_option("step_cap", int(os.environ.get("SAN_STEPS", "8")))
ctx.set_option("step_cap", int(os.environ.get("SAN_STEPS", "10")))
ctx.set_option("direct_after", 5)               # steps 1 .. 4: poisson_warm_kernel; 5 .. 9: poisson_direct_kernel
ctx.set_option("rows_wide_from_step", 5)        # steps 0 .. 4: 4-warp search; 5 .. 9: 8-warp search
ctx.set_option("match_win_until_step", 5)       # steps 0 .. 4: windowed matched solution (windows of 1024 nodes); 5 .. 9: one window
ctx.set_option("match_win_nodes", 1024)
for cfg in (0x111, 0x412):
    ctx.set_option("rows_cfg", cfg)
    r = ctx.solve_batch([D.Options(4, 11, 15.0, 0.002, 0.5, 0), D.Options(3, 11, 15.0, 0.002, 0.5, 1)], keep_steps=False)
    print("scf L11 rows_cfg", hex(cfg), [x.n_steps for x in r], r[0].Etotal, flush=True)
ctx.set_option("rows_cfg", 0x111)
r = ctx.solve_batch([D.Options(6, 12, 20.0, 0.001, 0.5, 0)], keep_steps=False)
print("scf L12", [x.n_steps for x in r], r[0].Etotal, flush=True)
ctx.set_option("direct_after", 2); ctx.set_option("step_cap", 5)
r = ctx.solve_batch([D.Options(3, 15, 20.0, 0.0003, 0.5, 0)], keep_steps=False)
print("scf L15 (chunked direct Poisson solve, windowed match)", [x.n_steps for x in r], r[0].Etotal, flush=True)
r = ctx.solve_batch([D.Options(10, 9, 15.0, 0.008, 0.5, 0)], keep_steps=False)
print("scf L9 (rows search on a coarse grid)", [x.n_steps for x in r], r[0].Etotal, flush=True)
L, delta, rmax = 10, 0.004, 15.0
N = (1 << L) + 1
rp = rmax / (np.exp((N - 1) * delta) - 1); rr = rp * (np.exp(np.arange(N) * delta) - 1)
V = np.zeros(N); V[1:] = -10.0 / rr[1:]
for impl in (4, 5, 6):
    s_, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, np.array([0, 1, 2, 3] * 8, np.int32), np.linspace(-40, -1, 32), np.full(32, 9, np.int32), impl=impl)
    print("lanes impl", impl, cnt[:8], flush=True)
