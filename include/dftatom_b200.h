/*
 * dftatom_b200 — C ABI of the B200-native radial Kohn-Sham SCF engine.
 *
 * Drop-in boundary for the computation behind aromanro/DFTAtom's
 *     static void DFT::DFTAtom::CalculateNonUniformLDA (int Z, int MultigridLevels, double alpha, double MaxR, double deltaGrid)
 *     static void DFT::DFTAtom::CalculateNonUniformLSDA(int Z, int MultigridLevels, double alpha, double MaxR, double deltaGrid)
 * (reference DFTAtom/DFTAtom.h:14,17; only call site DFTAtomFrame.cpp:190-195).  The reference has no
 * FFI / plugin interface: that static-function pair, selected by Options::method (Options.h:54), and the
 * text it prints on std::cout ARE the interface, so the entry points below carry the same arguments
 * (as `dftatom_options`, mirroring Options.h:48-54) and return the same numbers the text holds
 * (per-step eigenvalues + node counts + Etotal/Ekin/Ecoul/Eenuc/Exc, final configuration).
 *
 * Plain C: pointers and sizes only, no C++/torch types.  All floating point is IEEE FP64.
 * Every function returns 0 on success or a negative DFTATOM_E_* code; dftatom_last_error() gives text.
 * There is NO CPU fallback: without a CUDA device dftatom_create fails with DFTATOM_E_NO_DEVICE.
 */
#ifndef DFTATOM_B200_H
#define DFTATOM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DFTATOM_MAX_LEVELS 24          /* per spin channel; Z <= 118 needs 19 (SURVEY B.2) */
#define DFTATOM_MAX_STEPS_LDA 100      /* DFTAtom.cpp:396 */
#define DFTATOM_MAX_STEPS_LSDA 150     /* DFTAtom.cpp:908 */

enum {
    DFTATOM_OK = 0,
    DFTATOM_E_NO_DEVICE = -1,
    DFTATOM_E_BAD_OPTION = -2,         /* outside the ranges OptionsFrame.cpp:46,152-173 enforces */
    DFTATOM_E_MIXED_GRID = -3,         /* atoms of one batch must share (levels, delta, max_r) */
    DFTATOM_E_CUDA = -4,
    DFTATOM_E_ARG = -5
};

/* per-atom status (the reference is silent about non-convergence, DFTAtom.cpp:516-539; SURVEY §5) */
enum {
    DFTATOM_CONVERGED = 0,             /* the reference would have printed "Finished!" */
    DFTATOM_MAX_STEPS = 1,             /* step cap hit (100 LDA / 150 LSDA), like the reference's silent fall-through */
    DFTATOM_NUMERIC_FAILURE = 2        /* NaN/Inf in the energies */
};

/* Options.h:48-54 (field meaning identical; defaults Options.cpp:6: Z=36, levels=12, MaxR=10, delta=0.001, alpha=0.5, method=0) */
typedef struct {
    int Z;              /* 1..118 (OptionsFrame.cpp:152-154) */
    int levels;         /* MultigridLevels, N = 2^levels + 1 nodes; 8..20 accepted (dialog shows 10..20) */
    double max_r;       /* MaxR, 1..90 */
    double delta;       /* deltaGrid, (0,1] */
    double mixing;      /* alpha = weight of the OLD density, [0,1] */
    int method;         /* 0 = LDA (banner says "LSD"), 1 = LSDA */
} dftatom_options;

typedef struct {
    int n;              /* principal quantum number, 1-based as printed */
    int l;              /* 0..3 -> s p d f */
    int occ;            /* electrons in this (spin) subshell */
    int nodes;          /* n - l - 1, the "Num nodes" the reference prints */
    double E;           /* eigenvalue, Hartree */
} dftatom_level;

/* one "Step: k" block of the reference's output */
typedef struct {
    double E[2][DFTATOM_MAX_LEVELS];   /* eigenvalues, [spin][level in (n,l) order] */
    double Etotal, Ekin, Ecoul, Eenuc, Exc;
    int levels_converged;              /* reallyConverged of this step (DFTAtom.cpp:406,538) */
    int stop_criterion_met;            /* 1 if the "Finished!" test of DFTAtom.cpp:474 holds at this step (always the last step of a converged
                                          run; with set_option("run_to_cap", 1) the SCF continues past it and later steps may carry it too) */
} dftatom_step;

typedef struct {
    int status;                        /* DFTATOM_CONVERGED / MAX_STEPS / NUMERIC_FAILURE */
    int n_steps;                       /* number of "Step:" blocks = index of last step + 1 */
    int n_spin;                        /* 1 (LDA) or 2 (LSDA: alpha, beta) */
    int n_levels[2];
    dftatom_level levels[2][DFTATOM_MAX_LEVELS];   /* (n,l) order, eigenvalues of the last step */
    dftatom_level sorted[2][DFTATOM_MAX_LEVELS];   /* same, sorted by eigenvalue: the final "1s2 2s2 ..." line (DFTAtom.cpp:487-490) */
    double Etotal, Ekin, Ecoul, Eenuc, Exc;        /* last step */
} dftatom_result;

typedef struct dftatom_ctx dftatom_ctx;

/* ---- context ---- */
int dftatom_create(dftatom_ctx** ctx, int cuda_device);
void dftatom_destroy(dftatom_ctx* ctx);
const char* dftatom_last_error(void);
const char* dftatom_version(void);
/* tuning knobs (all default to reference-equivalent behaviour):
 *   "max_vcycles"  (default 8) V-cycles after the FMG ramp.  The reference runs 100 (PoissonSolver.h:117) because its
 *                   exit test err < 1e-14 never fires; the update norm reaches its FP64 rounding floor after ~6
 *                   (SURVEY fact 3).  A fixed, data-independent count keeps the solve a smooth function of the density,
 *                   which the SCF stop test |dE/E| < 1e-11 needs.  Set 100 to reproduce the reference's count.
 *   "refine_vcycles" (default 0 = off) V-cycles of an optional double-double defect correction after the plain solve.
 *                   It yields the discrete solution to FP64 representation accuracy, but the reference's own answer
 *                   carries the ~1e-9 rounding-floor bias of plain FP64 multigrid (worth ~1e-5 Ha in Etotal at Z~90),
 *                   so parity with the reference requires it to stay off.
 *   "vcycle_floor_stop" (default 0) 1 = stop as soon as the update norm stagnates (data dependent)
 *   "warm_start"   (default 1) from the second SCF step on, the first search round samples a geometric ladder of trial
 *                   energies around the previous step's eigenvalue (same root: the predicate is monotone); 0 = every
 *                   step searches [-Z^2-1, 50] from scratch like the reference
 *   "match_mode"   (default 0) 0 = segmented two-sided solve (production); 1 = serial reference-arithmetic kernel
 *   "search_kernel" (default 0) search_mode 0 on the logarithmic grid: 0 = lanes across the radial grid (numerov_rows.cu: one CTA per orbital,
 *                   128 radial segments, every thread 4 trial energies x 2 basis chains; 2-3 rounds of 4 energies per solve); 1 = lanes across 32 trial
 *                   energies (numerov_seg.cu / numerov_fast.cu, round 1's kernels; always used on the uniform grid).  "rows_cfg" (default 0x111):
 *                   groups of 4 trial energies per round of the rows kernel, one hex digit each (1, 2 or 4 = 128, 64 or 32 radial segments) for
 *                   untrusted ladders / trusted ladders / sectioning rounds
 *                   "rows_wide_from_step" (default 32; 0 = never): from this SCF step on an atom's orbitals are searched by the 8-warp shape of the
 *                   rows kernel (256 radial segments per orbital: half the depth of a round, for the steps where few atoms are left)
 *   "r_segments"   (default -1 = auto: 16 up to 16385 nodes, 32 above) search_kernel 1: radial segments per orbital of the parallel-in-r search
 *                   (one thread-block cluster per orbital); 0 = serial-in-r search only (one warp per orbital)
 *   "seg_threshold" (default 2400) search_kernel 1: the parallel-in-r search runs once at most this many orbitals are still active, the
 *                   serial-in-r one (fewer instructions, needs >= 4 warps per FP64 pipe to hide its dependent chain) above
 *   "search_mode"  (default 0) 0 = fused single-predicate multisection (production); 1 = reference-shaped three-stage
 *                   search (node-count window edges, then the sign change of y(0)), kept for validation
 *   "profile"      (default 0) time every kernel class with CUDA events, see dftatom_last_profile
 *   "stream_groups" (default 4; 1..8) a batch of >= 32 atoms on a grid of <= 16385 nodes is dealt into this many groups whose SCF chains run
 *                   concurrently on their own streams (atoms are independent; every launch of one chain depends on the previous one and most
 *                   are latency-bound: one group's Poisson solves overlap another's search).  Measured: C3 72.5 -> 66 ms.  Per-atom results do
 *                   not depend on it; the per-class CUDA-event times of "profile" then include the contention between the groups.
 *   "stream_poisson" (default 1) grids of at least "stream_min_levels" (default 15) levels with at least "stream_min_dens"
 *                   (default 4) densities in the batch: the Poisson solve runs as level visits streamed over all densities
 *                   (poisson_stream.cu: slab windows with halos, one launch per level visit) for the levels above
 *                   2^"stream_mid_levels" (default 11, 11..14) nodes and one CTA per density below, instead of one CTA / team
 *                   of CTAs per density for everything; 0 = never
 *   "poisson_exact" (default 0) 1 = bit-reproducible Poisson solve (poisson_exact.cu): the reference's FullCycle in the reference's own
 *                   floating-point operation order (no FMA), with its early exits and its 100 V-cycles; U(r) equals the CPU reference's
 *                   bit for bit (tests/test_gpu_components.py).  A parity / validation mode, ~50x slower than the production solver.
 *   "run_to_cap"   (default 0) 1 = the stop test of DFTAtom.cpp:474 is evaluated and recorded (dftatom_step.stop_criterion_met) but does
 *                   not end the SCF: every atom runs to the step cap.  Lets a test compare the record at the step where the REFERENCE
 *                   stopped, whatever step this implementation's own (noise-driven, DESIGN.md section 5) stop fires at.
 *   "adaptive_mixing" (default 0 = the reference's fixed linear mixing; results unchanged) 1 = opt-in damping beyond the reference: when an
 *                   atom's Etotal sloshes with period 2 (three changes of alternating sign decaying by less than 2x per step - the
 *                   nearly full nodeless 3d / 4f shells: Cu, Zn, Ho..Yb; the reference runs Er, Tm, Yb to its 100-step cap) the weight
 *                   of its old density is raised, alpha <- (1 + alpha) / 2, at most three times.  Lets all 92 atoms of the sweep converge.
 *   "use_graph"    (default 1) the steady-state SCF step is captured once into the body of a CUDA-graph WHILE node whose condition ("some
 *                   atom is still iterating") is set on the device (cudaGraphSetConditional): no host round trip between SCF steps.  Not used
 *                   with "profile" (per-class event timing needs host-side events between the launches), the validation search / match modes
 *                   and the cooperative team-mode Poisson kernel (one to three atoms on grids above 16385 nodes); 0 = host-driven loop.
 *   "use_pdl"      (default 1) the kernels of an SCF step are launched with programmatic stream serialization (each starts with
 *                   griddepcontrol.wait before its first global read): the next kernel's blocks are scheduled while the previous one drains.
 *                   Same records; 0 = plain stream order.
 *   "unit_guess"   (default 1) the Poisson solve of the SCF's start density (DFTAtom.cpp:371-392: a uniform sphere of Z electrons, boundary value Z -
 *                   linear in Z) is done once per grid for Z = 1 by the cold multigrid kernel and scaled per atom (grids up to 16385 nodes);
 *                   0 = one cold solve per atom and call.  Per-step parity with the reference unchanged (C3: 2.70e-6 vs 2.72e-6 Ha).
 *   "search_predict" (default 1) the production search starts every level of an SCF step from a ladder of 4 trial energies placed by what the
 *                   first steps of the reference's SCF are known to do: step 0 - hydrogenic levels of the initial potential (uniform sphere of
 *                   radius MaxR, DFTAtom.cpp:371-376: -Z^2/2n^2 + 3Z/(2 MaxR)); step 1 - one-sided (every level rises when the first real
 *                   density screens the nucleus); step 2 - default decay ratio of the shifts; later - extrapolated shift, offsets scaled
 *                   with the shifts.  0 = cold section of [-Z^2-1, 50] at step 0 and the plain previous-eigenvalue ladder.  Same results
 *                   (every bracket is certified by the Sturm count), fewer rounds.
 *   "graph_phases" (default 1) the graph loop is a chain of WHILE nodes, one per range of SCF steps between the step indices at which a
 *                   kernel shape hands over to another one ("rows_wide_from_step", "match_win_until_step"; all atoms of a batch step
 *                   together): every body holds only the shapes of its own range, no launch that returns at once.  0 = one WHILE node
 *                   whose body launches every shape at every step.  Same records either way.
 *   "step_cap"     (default 0 = the reference's caps, 100 LDA / 150 LSDA steps) a lower cap on the SCF steps of every atom of the batch
 *   "warm_vcycles" (default 7) / "warm_after" (default 1): from SCF step warm_after on the Poisson solve is warm_vcycles V-cycles in increment
 *                   form (A dU = -r 4 pi K (rho - rho_prev) from dU = 0, U += dU; "delta_poisson" 0 = iterate on U itself) instead of the full
 *                   multigrid cycle; warm_vcycles 0 = the full cycle at every step
 *   "warm_poisson" (default 1) those warm solves on grids of 2049 .. 16385 nodes by one CTA per density (poisson_warm.cu) while the atom's own
 *                   SCF step counter is below "warm_until_step" (default 32; 0 = always), by the cluster kernel below afterwards: both are
 *                   launched every step and the atom's step counter decides, so its records do not depend on what else is in the batch
 *   "coarse_exact" (default 1) warm solves: the levels below 2048 nodes (~60 latency-bound sweeps per V-cycle for a few hundred nodes) are
 *                   replaced by the exact solve of the 1024-node level's own equation (poisson_tri.cuh); 0 = swept like the reference does
 *   "direct_poisson" (default 1) warm solves in increment form from SCF step "direct_after" (default 4) on: the level-0 system of the increment
 *                   is solved directly (Thomas algorithm as block scans of affine maps, poisson_direct.cu; every grid of >= 2049 nodes) instead
 *                   of by V-cycles; the warm steps before it (large increments) and "direct_poisson" 0 use the V-cycle kernels above
 *   "recold_at"    (default -1 = never) this one SCF step solves the Poisson equation cold (full multigrid) again
 *   "match_win_until_step" (default 32; 0 = always one window) / "match_win_nodes" (default 8192): grids that fit one window of the matched-solution
 *                   kernel: while the atom's step counter is below the former its orbitals are solved in windows of the latter (3 CTAs per SM),
 *                   afterwards in one window (one CTA per SM, lowest latency)
 *   "cluster_poisson" (default 1) warm-started Poisson solves on grids of 2049 .. 16385 nodes run as one thread-block cluster of 8 CTAs per
 *                   density with the whole multigrid hierarchy in distributed shared memory (poisson_cluster.cu); 0 = one CTA per density.
 *                   "cluster_max_dens" (default: unlimited) restricts it to steps with at most that many atoms still iterating.
 *   "stream_variant" (default 0) window shape of the stream-mode Poisson visits: 0 = 256 threads x 16 nodes, 1 = 256 x 8, 2 = 512 x 8
 */
int dftatom_set_option(dftatom_ctx* ctx, const char* key, double value);

/* ---- L0 rules (host, integer) ---- */
/* AufbauPrinciple::GetSubshells + sort (AufbauPrinciple.h:36-75, DFTAtom.cpp:367). returns number of levels, or <0 */
int dftatom_aufbau(int Z, dftatom_level* out, int max_out);
/* DFTAtom::InitializeLevels (DFTAtom.cpp:611-638) */
int dftatom_split_spin(int Z, dftatom_level* alpha, int* n_alpha, dftatom_level* beta, int* n_beta, int* n_alpha_el, int* n_beta_el);
int dftatom_n_nodes(int levels);       /* PoissonSolver::GetNumberOfNodes, PoissonSolver.h:127-135 */

/* ---- sharding of a batch over GPUs (host; atoms are independent: one process per GPU, no collective, SURVEY 8e) ----
 * dftatom_estimate_cost: relative cost of one atom = its (spin) orbitals x the expected number of SCF steps (the nearly full nodeless
 * 3d / 4f shells - Cu, Zn, Ho..Yb - take 2-4x the steps of their neighbours).  dftatom_partition: longest-processing-time-first
 * assignment of n_atoms atoms to n_ranks ranks (rank_of[i] = rank of atom i; method may be NULL = LDA); deterministic.  The estimate
 * only balances the shards: results never depend on it. */
double dftatom_estimate_cost(int Z, int method);
int dftatom_partition(const int* Z, const int* method, int n_atoms, int n_ranks, int* rank_of);

/* ---- L2: the SCF (replaces CalculateNonUniformLDA/LSDA for a whole batch of independent atoms) ----
 * opts[n_atoms], out[n_atoms] are HOST arrays.  steps may be NULL; otherwise it is a HOST array of
 * n_atoms * steps_stride records receiving every SCF step (record k of atom a at steps[a*steps_stride + k]).
 * All atoms of one call must share (levels, delta, max_r); Z, mixing, method may differ. */
int dftatom_solve_batch(dftatom_ctx* ctx, const dftatom_options* opts, int n_atoms, dftatom_result* out,
                        dftatom_step* steps, int steps_stride);

/* ---- L2 with the converged radial state ----
 * dftatom_solve_batch_radial = dftatom_solve_batch plus, when `radial` is not NULL, the radial arrays of every atom copied into the
 * caller's HOST arrays below (dftatom_solve_batch is this call with radial == NULL).  Every pointer may be NULL: that array is not
 * exported.  N = dftatom_n_nodes(levels); atoms are indexed in call order.
 *
 * What the arrays hold: the state of the atom's LAST SCF step, in the reference's loop order (DFTAtom.cpp:396-481 / :908-1006) - the
 * orbitals were solved in the potential of the step before, `rho` is the mixed density of the last step, and `v` / `v_hartree` were
 * computed from that rho.  These are the arrays the reference holds when its loop ends (the oracle's orc_scf_ex exports the same).  An
 * atom that stopped keeps them frozen while the rest of the batch iterates (every SCF kernel returns at once for a finished atom), so
 * they do not depend on what else is in the batch.
 *
 * Orbitals: u_nl(r) = r R_nl(r), the u whose square the density accumulates (u_i = y_i e^{i delta/2} / sqrt(integral of u^2 dr) on the
 * logarithmic grid, DFTAtom.cpp:36-56; y_i / sqrt(...) on the uniform grid), normalised so that sum_i wjac_i u_i^2 = 1 with the Simpson38
 * weights times the jacobian that the energies use (Integral.h:50-73 x DFTAtom.cpp:47,442).  The sign is fixed so that u > 0 at the
 * first node away from the nucleus (u ~ r^{l+1}).  Node 0 (r = 0) holds 0 in every exported array (the SCF arrays hold 0 there).  The
 * last node holds the orbital's value and is part of its normalisation; the density, like the reference's (DFTAtom.cpp:558-559), sums
 * occ u^2 / (4 pi r^2) over nodes 1 .. N-2 only.
 * Rows: atoms in call order, then spin (alpha, beta), then the (n, l) order of dftatom_result.levels; an atom has as many rows as
 * dftatom_aufbau (LDA) or dftatom_split_spin (n_alpha + n_beta levels, LSDA) gives it.  An `orbital_rows` smaller than the batch needs
 * (when `orbitals` or `moments` is given) returns DFTATOM_E_ARG before anything is solved.
 * Moments: sum_i wjac_i u_i^2 f(r_i) for f = 1/r (node 0 left out), r, r^2 - <1/r>, <r>, <r^2> of the normalised orbital.
 * atom_moments: sum_i wjac_i 4 pi r_i^2 rho_i (the electron count) and sum_i wjac_i 4 pi r_i^4 rho_i (<r^2> summed over the electrons),
 * rho = the total density.
 * The export runs after the SCF loop: its kernels and copies are not part of dftatom_last_timing; its bytes are part of the d2h count of
 * dftatom_last_transfer. */
#define DFTATOM_N_MOMENTS 3            /* <1/r>, <r>, <r^2> */
typedef struct {                       /* HOST pointers; any may be NULL (not exported) */
    double* r;                         /* [N] grid nodes r_i */
    double* rho;                       /* [n_atoms][2][N] density per spin (LDA: row 0 = total density, row 1 = 0) */
    double* v;                         /* [n_atoms][2][N] Kohn-Sham potential per spin (LDA: row 1 = 0) */
    double* v_hartree;                 /* [n_atoms][N] V_H = U / r */
    double* orbitals;                  /* [orbital_rows][N] u_nl(r), rows as described above */
    long long orbital_rows;            /* capacity of `orbitals` / `moments` in rows */
    double* moments;                   /* [orbital_rows][DFTATOM_N_MOMENTS] */
    double* atom_moments;              /* [n_atoms][2]: electron count, <r^2> of the total density */
} dftatom_radial;
int dftatom_solve_batch_radial(dftatom_ctx* ctx, const dftatom_options* opts, int n_atoms, dftatom_result* out, dftatom_step* steps,
                               int steps_stride, const dftatom_radial* radial);
/* The moment reduction of the export on caller-supplied orbitals u[n_rows][N] (HOST) of the grid (levels, delta, max_r; delta = 0: the
 * uniform grid): moments[n_rows][DFTATOM_N_MOMENTS] = sum_i wjac_i u_i^2 f(r_i), f = 1/r (node 0 left out), r, r^2.  The rows are used
 * as given (no normalisation, no sign). */
int dftatom_radial_moments(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* u, int n_rows, double* moments);

/* device time (ms, CUDA events) of the last solve_batch's SCF loop, and number of kernel launches it issued */
int dftatom_last_timing(dftatom_ctx* ctx, double* device_ms, long long* kernel_launches);
/* bytes the last solve_batch copied host -> device (atom / orbital descriptors; grid tables are cached per context and not counted)
 * and device -> host (per-atom state + step records: every step when `steps` was given, else the last record of every atom) */
int dftatom_last_transfer(dftatom_ctx* ctx, long long* h2d_bytes, long long* d2h_bytes);
/* number of SCF steps the last solve_batch ran inside the CUDA-graph WHILE node (set_option "use_graph", default 1: from step "warm_after" on
 * the whole SCF loop of the batch is ONE graph launch whose loop condition is evaluated on the device; 0 = the host enqueued every step) */
int dftatom_last_graph_iterations(dftatom_ctx* ctx, long long* iterations);

/* Per-kernel-class profile of the last solve_batch, filled when set_option("profile", 1) was on: device time of
 * every launch of the class (CUDA events on the launching stream), launch count and algorithmic work
 * (class 0: Numerov (lane, node-step) pairs; class 3: Gauss-Seidel node-updates; others: 0). */
enum { DFTATOM_K_SEARCH = 0, DFTATOM_K_MATCH = 1, DFTATOM_K_DENSITY = 2, DFTATOM_K_POISSON = 3, DFTATOM_K_POTENTIAL = 4, DFTATOM_K_COUNT = 5 };
/* work: search = (lane, node-step) pairs of the shooting sweeps; match = orbital solves; density = search rounds summed over the
   orbital solves; poisson = Gauss-Seidel node updates; potential = 0 */
typedef struct { double ms; long long launches; double work; } dftatom_kernel_profile;
int dftatom_last_profile(dftatom_ctx* ctx, dftatom_kernel_profile* out /* [DFTATOM_K_COUNT] */);
/* measured FP64 FMA peak of the device (TFLOP/s, 2 flops per DFMA), the roofline denominator of the shooting kernel */
int dftatom_measure_fp64_peak(dftatom_ctx* ctx, double* tflops);

/* ---- L1 component entry points (HOST buffers; used by the parity tests and the microbenches) ---- */

/* Batched inward Numerov sweeps on one potential (Numerov.h:272-349 CountNodes and :351-401 SolutionInZero).
 * V[n_nodes] potential on the log grid, lanes k = 0..n_lanes-1 with (l[k], E[k], nodes_limit[k]).
 * y0_sign[k] = 1 if SolutionInZero > 0 else 0; y0_log2[k] ~ log2|y0| (for the 1e15 guard).
 * impl = 1: reference-shaped sweep, count[k] = CountNodes (with its early exits, clamped at nodes_limit+1).
 * impl = 0: the production tile-staged sweep, count[k] = number of ALL sign changes of y_start..y_1,y_0 (the Sturm count
 *           the fused search uses; nodes_limit ignored; -1 if the lane hit a non-positive 1 - f/12).
 * impl = 2: the same count through the parallel-in-r sweep (one thread-block cluster per 32 lanes, warp = radial segment,
 *           set_option("r_segments") segments).
 * impl = 3: count[k] = SolveSchrodingerCountNodesFromNucleus (Numerov.h:204-270: the OUTWARD sweep from the nucleus with its early exits -
 *           overflow, count > nodes_limit, outer classical turning point; public in the reference but without a caller); y0_* are 0.
 * impl = 4, 5, 6: the count of impl 0 through the production sweep of the SCF search (numerov_rows.cu: lanes across the radial grid, every
 *           thread 4 trial energies x 2 basis chains): 4 energies on 128 radial segments, 8 on 64, 16 on 32 per CTA (logarithmic grid only). */
int dftatom_numerov_lanes(dftatom_ctx* ctx, const double* V, int levels, double delta, double max_r, int n_lanes,
                          const int* l, const double* E, const int* nodes_limit, int impl,
                          int* y0_sign, double* y0_log2, int* count);
/* the same, plus a device-timed repetition for the C5b microbench: after the checked launch the kernel is launched `reps` more
 * times between CUDA events (potential table and lanes resident in HBM); ms_per_launch = their average,
 * lane_node_steps = sum over lanes of (cut-off index - 1), the node-steps one launch performs (SURVEY 8d: 11 FLOP each) */
int dftatom_numerov_lanes_timed(dftatom_ctx* ctx, const double* V, int levels, double delta, double max_r, int n_lanes,
                                const int* l, const double* E, const int* nodes_limit, int impl,
                                int* y0_sign, double* y0_log2, int* count, int reps, float* ms_per_launch, double* lane_node_steps);
/* per-level eigenvalue search on one potential (DFTAtom.cpp:497-541 + LocateInterval :566-604), all levels concurrently */
int dftatom_level_search(dftatom_ctx* ctx, const double* V, int levels, double delta, double max_r, int Z,
                         int n_levels, const int* n, const int* l, double* E_out, int* converged_out);
/* two-sided matched + normalised solution u(r) (Numerov.h:403-504 + DFTAtom.cpp:36-56) */
int dftatom_numerov_orbital(dftatom_ctx* ctx, const double* V, int levels, double delta, double max_r,
                            int l, double E, double* u_out, int* match_point);
/* SolvePoissonNonUniform (PoissonSolver.h:51-81) for n_dens densities rho[n_dens][N] with boundary values (0, Z[k]) */
int dftatom_poisson_solve(dftatom_ctx* ctx, int levels, double delta, double max_r, int n_dens, const int* Z,
                          const double* rho, double* U, int* vcycles_used);
/* n_cycles reference-shaped V-cycles (PoissonSolver.h:155-159) in place on phi[n_dens][N] with source src[n_dens][N] */
int dftatom_poisson_vcycles(dftatom_ctx* ctx, int levels, double delta, int n_dens, double* phi, const double* src,
                            int n_cycles, double* last_err);
/* VWNExchCor::Vexc / eexcDif, LDA (VWNExcCor.h:73-128) and LSDA (:134-312; pass rho_b != NULL) */
int dftatom_vwn(dftatom_ctx* ctx, int n, const double* rho_a, const double* rho_b, double* va, double* vb,
                double* vexc, double* eexcdif);
/* LDA exchange-correlation by functional: 0 = VWN (= dftatom_vwn, the one the reference's SCF uses), 1 = Chachiyo (ExcCor.h:27-95 with
 * the parameters of :12-17), 2 = Chachiyo improved (:20-25).  The Chachiyo functionals are reachable from no option of the reference. */
int dftatom_xc_lda(dftatom_ctx* ctx, int functional, int n, const double* rho, double* vexc, double* eexcdif);
/* Integral::Simpson38 (Integral.h:50-73) of n_rows rows of length n */
int dftatom_simpson38(dftatom_ctx* ctx, double step, const double* v, int n, int n_rows, double* out);

/* The whole quadrature family of Integral.h as block reductions: rule 0 Trapezoid (Integral.h:11-23), 1 SimpsonOneThird (:25-48),
 * 2 Simpson38 (:50-73, the only one the reference's SCF calls), 3 Boole (:75-104), 4 Romberg (:106-155, err 1e-18, minSteps 3).
 * n must satisfy the reference's assertions for the rule (odd / 4k+1 ...), else DFTATOM_E_ARG. */
int dftatom_integrate(dftatom_ctx* ctx, int rule, double step, const double* v, int n, int n_rows, double* out);

/* ---- microbenches on DEVICE-resident data (bench.py `value` legs); pointers are CUDA device addresses ---- */
/* Stream-mode V-cycles (config C5a: many densities on a grid that does not fit on chip; levels >= 15).  n_cycles V-cycles
 * (PoissonSolver.h:155-159: 3 + 3 Gauss-Seidel sweeps per level, injection of the residual, linear prolongation) in place on
 * d_phi[n_dens][ld] with source d_src[n_dens][ld] (natural node order, N = 2^levels + 1 <= ld, ld even, both 16-byte aligned).
 * d_scratch: dftatom_poisson_scratch_bytes(levels, n_dens) bytes.  fuse_tops != 0: the last visit of level 0 of one cycle and
 * the first visit of the next are one pass over the level (6 sweeps).  device_ms: CUDA-event time of the n_cycles cycles;
 * kernel_launches: launches issued.  The call returns after the work has completed. */
int dftatom_poisson_vcycles_dev(dftatom_ctx* ctx, int levels, double delta, int n_dens, void* d_phi, const void* d_src, long long ld,
                                void* d_scratch, long long scratch_bytes, int n_cycles, int fuse_tops, float* device_ms,
                                long long* kernel_launches);
long long dftatom_poisson_scratch_bytes(int levels, int n_dens);

#ifdef __cplusplus
}
#endif
#endif
