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
    int occ;            /* electrons in this (spin) subshell; for an atom solved with a configuration (dftatom_solve_batch_config) the
                           occupation rounded to the nearest integer - the exact value is the caller's entry with the same (n, l, spin) */
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
 *   "unit_guess"   (default 1) the Poisson solve of the SCF's start density (DFTAtom.cpp:371-392: a uniform sphere of Q electrons, boundary value Q -
 *                   linear in the electron count Q, = Z for the neutral atom) is done once per grid for Q = 1 by the cold multigrid kernel and scaled
 *                   per atom (grids up to 16385 nodes);
 *                   0 = one cold solve per atom and call.  Per-step parity with the reference unchanged (C3: 2.70e-6 vs 2.72e-6 Ha).
 *   "search_predict" (default 1) the production search starts every level of an SCF step from a ladder of 4 trial energies placed by what the
 *                   first steps of the reference's SCF are known to do: step 0 - hydrogenic levels of the initial potential (uniform sphere of
 *                   radius MaxR, DFTAtom.cpp:371-376: -Z^2/2n^2 + 3Q/(2 MaxR), Q = the electron count); step 1 - one-sided (every level rises when the first real
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
 *                   multigrid cycle; warm_vcycles 0 = the full cycle at every step.  On grids of 2049 .. 16385 nodes these V-cycles are run
 *                   by one CTA per density (poisson_warm.cu), the levels below 2048 nodes (~60 latency-bound sweeps per V-cycle for a few
 *                   hundred nodes) replaced by the exact solve of the 1024-node level's own equation (poisson_tri.cuh)
 *   "direct_poisson" (default 1) warm solves in increment form from SCF step "direct_after" (default 4) on: the level-0 system of the increment
 *                   is solved directly (Thomas algorithm as block scans of affine maps, poisson_direct.cu; every grid of >= 2049 nodes) instead
 *                   of by V-cycles; the warm steps before it (large increments) and "direct_poisson" 0 use the V-cycles above
 *   "match_win_until_step" (default 32; 0 = always one window) / "match_win_nodes" (default 8192): grids that fit one window of the matched-solution
 *                   kernel: while the atom's step counter is below the former its orbitals are solved in windows of the latter (3 CTAs per SM),
 *                   afterwards in one window (one CTA per SM, lowest latency)
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
 * dftatom_aufbau (LDA) or dftatom_split_spin (n_alpha + n_beta levels, LSDA) gives it, a configured atom (dftatom_solve_batch_config) as
 * many as its configuration has entries.  An `orbital_rows` smaller than the batch needs
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
/* ---- L2 with electron configurations: ions, excited states, empty channels, fractional occupations ----
 * A configuration is a list of orbitals (n, l, spin, occ), occ a double.  Every entry is one orbital the SCF solves (node count
 * n - l - 1); occ = 0: the orbital is solved, reported and exported, but adds nothing to the density or to E_el = sum occ eps.
 *   LDA  (methods 0, 2): spin = 0 and 0 <= occ <= 2 (2l + 1).   LSDA (methods 1, 3): spin = 0 (alpha) or 1 (beta), 0 <= occ <= 2l + 1.
 *   1 <= n <= 8, 0 <= l <= min(3, n - 1); no duplicate (n, l, spin); at most DFTATOM_MAX_LEVELS entries per spin and at least one alpha
 *   entry; every occ finite; the electron count Q = sum occ satisfies 0 < Q <= Z + 2.
 * A violation returns DFTATOM_E_BAD_OPTION (the message names the atom and the entry) before anything is solved.  The entries of each
 * spin are solved, reported (dftatom_result.levels, dftatom_step.E) and exported (radial rows) in (n, l) order, the order of
 * dftatom_aufbau.  What depends on Q: the start density (a uniform sphere of Q_s electrons per spin) and the Hartree boundary value
 * U(Rmax) = Q.  The nuclear charge stays Z: V = (-Z + U) / r, the energies, the search bracket [-Z^2 - 1, 50]. */
typedef struct { int n, l, spin; double occ; } dftatom_occupation;
typedef struct { int n_orbitals; dftatom_occupation orb[2 * DFTATOM_MAX_LEVELS]; } dftatom_config;
/* The reference's configuration of atom Z (dftatom_aufbau / dftatom_split_spin: the same entries, empty beta levels omitted) ionised by
 * `charge` electrons (may be fractional; < 0 = anion), alpha entries then beta entries, each in (n, l) order.
 *   Cations lose electrons from the occupied subshell of largest n, among those of largest l, one subshell at a time (an emptied subshell
 *   is dropped): Fe2+ = [Ar] 3d6, Cr+ = [Ar] 3d4 4s1 (the reference's Aufbau keeps Cr 3d4 4s2), Cu+ = [Ar] 3d9 4s1 (its Cu is 3d9 4s2;
 *   pass [Ar] 3d10 explicitly for the other one).
 *   Anions gain electrons in the reference's filling (Madelung) order from the first subshell that is not full: O- = 2p5, Ne- = ... 3s1.
 *   LSDA: every subshell's total is split like dftatom_split_spin: alpha min(occ, 2l + 1), beta the rest, listed only when nonzero.
 * charge == 0 reproduces dftatom_aufbau / dftatom_split_spin exactly.  -2 <= charge < Z, else DFTATOM_E_BAD_OPTION. */
int dftatom_config_aufbau(int Z, int method, double charge, dftatom_config* out);
/* = dftatom_solve_batch_radial with per-atom configurations: configs == NULL or configs[a].n_orbitals == 0: the Aufbau atom (bit for bit
 * the result of dftatom_solve_batch_radial, which is this call with configs == NULL).  The radial export's rows of a configured atom are
 * its configured entries. */
int dftatom_solve_batch_config(dftatom_ctx* ctx, const dftatom_options* opts, const dftatom_config* configs, int n_atoms,
                               dftatom_result* out, dftatom_step* steps, int steps_stride, const dftatom_radial* radial);
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
/* Logarithmic derivatives D_l(E) = u'(r_c) / u(r_c) of the radial solution regular at the nucleus, for every (channel, energy) pair:
 * the transferability diagnostic of pseudopotential generation, and the norm-conservation identity dD/dE = -2 int_0^rc u^2 dr / u(r_c)^2.
 * Grid (levels, delta, max_r) as in the other component entries (delta = 0: the uniform grid of methods 2 / 3), N = 2^levels + 1.
 * V[n_pot][N] HOST potentials (Hartree; node 0 ignored), e.g. rows of dftatom_radial.v.  Channel c = (V row pot[c], l[c], radius r_c[c]
 * in bohr); E[n_energies] HOST energies shared by all channels, in any order.  out[n_channels][n_energies]; r_used[n_channels] (may be
 * NULL) receives the radius actually used, the node r_(i_c) nearest to r_c[c].
 * Definition: g_i = f_i / 12 = (2 K_i (V_i - E) + K_i l(l+1) / r_i^2 + delta^2 / 4) / 12, K_i = (Rp delta e^(delta i))^2 (uniform grid:
 * K = h^2, no delta^2 / 4 term).  The outward Numerov solution starts from y_0 = 0, y_1 = r_1^(l+1) e^(-delta/2) (uniform grid: h^(l+1))
 * and steps w_(i+1) = 2 w_i - w_(i-1) + 12 g_i y_i, w = (1 - g) y, through every turning point to i_c + 1; u = y e^(delta i / 2)
 * (uniform grid: u = y).  u'(r_c) from the fourth-order index derivative y'_i = [(1 - 2 g_(i+1)) y_(i+1) - (1 - 2 g_(i-1)) y_(i-1)] / 2.
 * int_0^rc u^2 dr by Simpson's 1/3 rule on nodes 0..i_c times dr/di (3/8 rule on the last three intervals when i_c is odd).
 *   D      u'(r_c) / u(r_c), bohr^-1
 *   u, du  u(r_c) and u'(r_c) of the solution scaled to int_0^rc u^2 dr = 1, u > 0 next to the nucleus
 *   nodes  sign changes among the non-zero values of y_1 .. y_(i_c); the phase pi nodes - atan(r_c D) is continuous and increasing in E
 * A lane whose grid is too coarse (1 - g_i <= 0 at some node 2 <= i <= i_c + 1) returns nodes = -1 and NaN in D, u, du.  Every other lane
 * returns finite values (the sweep is rescaled by powers of two).
 * Validation before anything runs on the device: a bad grid returns DFTATOM_E_BAD_OPTION; n_pot, n_channels, n_energies >= 1,
 * 0 <= pot < n_pot, 0 <= l <= 3, r_2 <= r_c <= r_(N-2), every E finite and V finite at nodes 1..N-1, else DFTATOM_E_ARG naming the
 * channel, energy or potential row. */
typedef struct { double D, u, du; int nodes, pad; } dftatom_logderiv;      /* 32 bytes */
int dftatom_log_derivatives(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* V, int n_pot,
                            const int* pot, const int* l, const double* r_c, int n_channels,
                            const double* E, int n_energies, dftatom_logderiv* out, double* r_used);
/* Troullier-Martins norm-conserving pseudization of all-electron valence orbitals, and unscreening to ionic semilocal potentials.
 * Grid (levels, delta, max_r) and r_c rounding (the nearest node i_c, ties to the inner node), quadrature (Simpson 1/3 on nodes 0..i_c,
 * the 3/8 rule on the last three intervals when i_c is odd) and outward sweep are those of dftatom_log_derivatives.
 * V[n_pot][N] HOST potentials (node 0 ignored), u[n_orb][N] HOST all-electron orbitals u_nl(r) (e.g. rows of dftatom_radial.v and
 * dftatom_radial.orbitals).  Channel c = ch[c]: potential row pot, orbital row orbital, l, eigenvalue eps, occupation occ, radius r_c.
 * AE data at r_c: the sweep at E = eps on V[pot] gives D = u'/u and u_n(r_c) (solution normalised to int_0^rc u^2 dr = 1); a = |u(i_c)|,
 * s = sign u(i_c), q = a^2 / u_n(r_c)^2 (the AE norm inside r_c); V' and V'' at r_c from 5-point central differences in the index with
 * the chain rule: V' = V_i / J, V'' = (V_ii - delta V_i) / J^2, J = dr/di = delta (r + Rp) (uniform grid: J = h).
 * Pseudo-orbital inside r_c: u_ps = r^(l+1) e^p(r), p = c0 + c2 r^2 + c4 r^4 + ... + c12 r^12, with
 *   p = ln(a / r_c^(l+1)),  p' = D - (l+1)/r,  p'' = 2(V - eps) - 2(l+1)p'/r - p'^2,
 *   p''' = 2V' + 2(l+1)p'/r^2 - 2(l+1)p''/r - 2p'p'',
 *   p'''' = 2V'' - 4(l+1)p'/r^3 + 4(l+1)p''/r^2 - 2(l+1)p'''/r - 2p''^2 - 2p'p'''   at r_c,
 *   c2^2 + (2l+5) c4 = 0 (V_scr''(0) = 0), and the norm F(c2) = ln S(c2) - ln q = 0, S = Simpson sum of r^(2l+2) e^(2p) dr/di over 0..i_c.
 * For a given c2 the derivative conditions are linear in c6..c12.  Root: with x = c2 r_c^2 the ladder x = +-k/2 (k = 0..128) is scanned
 * outward from 0, the negative interval first at each |x|; the root in the first interval where F changes sign, to 1e-13 relative in c2.
 * out[c]: c0, c2, ..., c12 (bohr^-2k), r_c used, q, status: 0 ok, 1 no sign change on the ladder, 2 the sweep met 1 - g <= 0 (q = NaN),
 * 3 the multisection stopped short of 1e-13 (no sub-interval of the bracket changed sign, e.g. F not finite inside it, or 40 rounds).
 * Rows (each output may be NULL), node 0 = 0 in every row:
 *   u_ps[n_channels][N]   r^(l+1) e^p for i <= i_c, s u(i) copied for i > i_c
 *   v_scr[n_channels][N]  eps + [p'' + p'^2 + 2(l+1) p'/r] / 2 for i <= i_c (p'/r a polynomial), V[pot] copied for i > i_c
 *   rho_val[n_pot][N]     valence density sum occ u_ps^2 / (4 pi r^2) of the channels sharing the row (0 for a row without channels)
 *   v_ion[n_channels][N]  V_scr - V_H - V_xc: V_H = U / r from the cold Poisson solve of rho_val with boundary value Q_v = sum occ
 *                         (V_H = 0 when Q_v = 0), V_xc the spin-unpolarised VWN LDA of the SCF
 * A failed channel (status != 0) has NaN coefficients and NaN in u_ps, v_scr at nodes 1..i_c; its row's rho_val and every v_ion row of
 * that potential row are NaN at nodes 1..N-1.
 * Validation before anything runs on the device (outputs untouched): a bad grid returns DFTATOM_E_BAD_OPTION; DFTATOM_E_ARG, naming the
 * channel or row, for NULL V, u, ch or out, n_pot, n_orb or n_channels < 1, pot or orbital out of range, l outside 0..3, two channels of
 * one pot with the same l, r_c outside [r_3, r_(N-3)] (the 5-point stencil at i_c stays off node 0), eps not finite, occ not finite or outside [0, 2(2l+1)], V or u not finite at
 * nodes 1..N-1, u(i_c) = 0, or a sign change among the non-zero values of u at nodes i_c..N-1 (r_c inside the outermost node). */
typedef struct { int pot, orbital, l, pad; double eps, occ, r_c; } dftatom_tm_channel;      /* 40 bytes */
typedef struct { double c[7], r_c, q; int status, pad; } dftatom_tm_result;               /* 80 bytes */
int dftatom_tm_pseudize(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* V, int n_pot, const double* u, int n_orb,
                        const dftatom_tm_channel* ch, int n_channels, dftatom_tm_result* out, double* u_ps, double* v_scr,
                        double* v_ion, double* rho_val);
/* Nonlinear core correction (Louie, Froyen and Cohen 1982): the core density, its partial core, and the unscreening with it.
 * Grid (levels, delta, max_r; delta = 0: uniform), rounding to the nearest node (ties to the inner one) and the index derivative with
 * J = dr/di = delta (r + Rp) (uniform grid: J = h) are those of dftatom_tm_pseudize.
 * u[n_orb][N] HOST all-electron orbitals.  Core entry k = core[k]: output row `row`, orbital row `orbital`, occupation occ.
 *   rho_core[p] = sum occ u^2 / (4 pi r^2) over the entries of row p at nodes 1..N-2 (the SCF's density convention), 0 at nodes 0, N-1.
 * Partial core of row p with radius r_pc[p] >= 0:
 *   r_pc = 0: the full core, rho_pc = rho_core, i_pc = 0, A = B = 0.
 *   else i_pc = the nearest node, rho = rho_core(i_pc), rho' = its 5-point index derivative / J, t = 1 + r rho' / rho at r = r_(i_pc);
 *   x the root in (0, pi) of x cos x - t sin x = 0 (unique for t < 1: x cot x falls from 1 to -inf), found by bisection to the last
 *   bit; B = x / r, A = rho r / sin x; rho_pc = A sin(B r_i) / r_i for 1 <= i < i_pc, rho_core for i >= i_pc, 0 at node 0 (value and
 *   slope of rho_core at r_pc).
 * out[p]: r_pc used (the node radius, 0 for the full core), A, B, n_core = sum wjac 4 pi r^2 rho_core, n_pc likewise of rho_pc (wjac the
 * weights of the radial export), i_pc, status: 0 ok, 1 rho <= 0 or t >= 1 (the core density does not decrease at r_pc): A, B and
 * rho_pc at nodes 1..N-1 NaN.  rho_core, rho_pc [n_rows][N] may be NULL.
 * Validation before anything runs on the device (outputs untouched): a bad grid returns DFTATOM_E_BAD_OPTION; DFTATOM_E_ARG, naming the
 * row or entry, for NULL u, r_pc or out (core with n_core > 0), n_orb or n_rows < 1, n_core < 0, r_pc not finite, negative, in (0, r_3)
 * or above r_(N-3), an entry's row or orbital out of range, occ not finite or outside [0, 14], u not finite at nodes 1..N-1. */
typedef struct { int row, orbital; double occ; } dftatom_core_orbital;                                     /* 16 bytes */
typedef struct { double r_pc, A, B, n_core, n_pc; int i_pc, status, pad; } dftatom_pcc_result;           /* 56 bytes */
int dftatom_partial_core(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* u, int n_orb, const dftatom_core_orbital* core,
                         int n_core, const double* r_pc, int n_rows, dftatom_pcc_result* out, double* rho_core, double* rho_pc);
/* dftatom_tm_pseudize with the core-corrected unscreening V_ion,l = V_scr,l - V_H[rho_val] - V_xc(rho_val + rho_pc): rho_pc[n_pot][N]
 * HOST, one row per potential row (e.g. of dftatom_partial_core); V_H and rho_val stay those of the valence density.  rho_pc = NULL is
 * dftatom_tm_pseudize.  Validation adds DFTATOM_E_ARG for a rho_pc row that is not finite or negative at nodes 1..N-1. */
int dftatom_tm_pseudize_core(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* V, int n_pot, const double* u, int n_orb,
                             const dftatom_tm_channel* ch, int n_channels, dftatom_tm_result* out, double* u_ps, double* v_scr,
                             double* v_ion, double* rho_val, const double* rho_pc);
/* Kleinman-Bylander (KB) form of semilocal pseudopotentials: one local potential plus one separable projector per other channel,
 * V_NL = |beta> E_KB <beta|, with the Gonze-Stumpf-Scheffler (GSS) ghost-state test.  Grid (levels, delta, max_r) and the "sweep rule on
 * 0..n" (Simpson 1/3 on nodes 0..m, the 3/8 rule on the last three intervals when n is odd, times dr/di) are those of
 * dftatom_log_derivatives / dftatom_tm_pseudize.
 * V[n_rows][N] HOST screened potentials (node 0 ignored), u[n_rows][N] HOST pseudo-orbitals, e.g. v_scr and u_ps of dftatom_tm_pseudize.
 * Channel c = ch[c]: projects V[row] against the local potential V[loc] at angular momentum l, reference eigenvalue eps.
 *   dV_i = V[row]_i - V[loc]_i (nodes >= 1); i_s = the largest node with dV_i != 0 (0 if none), r_s = r_(i_s)
 *   a = sum w_i u_i^2 dV_i, b = sum w_i u_i^2 dV_i^2 (sweep rule on 0..i_s); E_KB = b / a; cos = a / sqrt(<u|u> b), <u|u> = sum over all
 *   nodes of the wjac weights of the radial export times u^2; beta_i = dV_i u_i / sqrt(b) (sum w beta^2 = 1 with the same rule)
 *   eps_loc[0], eps_loc[1]: the eigenvalues with 0 and 1 nodes of -1/2 u'' + [V[loc] + l(l+1)/2r^2] u in the box u(max_r) = 0, found by
 *   the energy search of the SCF (dftatom_level_search) with the bracket bottom -Z_b^2 - 1, Z_b the smallest integer >= 1 with
 *   -Z_b^2 - 1 <= min over nodes 1..N-1 of V[loc] (Z_b > 118: DFTATOM_E_ARG, "local potential too deep")
 *   ghost (GSS, nodeless reference state): E_KB > 0: 1 iff eps > eps_loc[1]; E_KB < 0: 1 iff eps > eps_loc[0]; else 0
 *   status: 0 ok; 1 local channel (row == loc): beta = 0, E_KB = 0, cos = 1, ghost = 0, eps_loc NaN; 2 a = 0 or i_s < 3: E_KB and cos
 *   NaN, beta = 0, ghost = -1; 3 the search did not converge for eps_loc[0] or [1]: eps_loc holds what it found, ghost = -1
 * beta[n_channels][N] (may be NULL): the projectors, 0 outside nodes 1..i_s.
 * Validation before anything runs on the device (outputs untouched): a bad grid returns DFTATOM_E_BAD_OPTION; DFTATOM_E_ARG, naming the
 * channel or row, for NULL V, u, ch or out, n_rows or n_channels < 1, row or loc out of range, l outside 0..3, eps not finite, V or u
 * not finite at nodes 1..N-1, i_s > N - 3, or a local potential too deep. */
typedef struct { int row, loc, l, pad; double eps; } dftatom_kb_channel;                                   /* 24 bytes */
typedef struct { double E_KB, cos, eps_loc[2], r_s; int i_s, ghost, status, pad; } dftatom_kb_result;     /* 56 bytes */
int dftatom_kb_form(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* V, const double* u, int n_rows,
                    const dftatom_kb_channel* ch, int n_channels, dftatom_kb_result* out, double* beta);
/* Logarithmic derivatives of the KB Hamiltonian: the solution regular at the nucleus of
 *   -1/2 u'' + [V_loc + l(l+1)/2r^2 - E] u + E_KB beta <beta|u> = 0
 * for every (channel, energy).  V_loc[n_pot][N] HOST local potentials, beta[n_proj][N] HOST projectors (e.g. of dftatom_kb_form),
 * channel c = ch[c]: potential row pot, projector proj (-1: none), l, E_KB, radius r_c.  E, out, r_used, the rounding of r_c and the
 * meaning of D, u, du and nodes are those of dftatom_log_derivatives; a channel with proj = -1 is computed by its sweep (bit for bit).
 * With a projector: u_h = the outward homogeneous solution of dftatom_log_derivatives; u_p = the outward solution driven by -beta, from
 * y_0 = y_1 = 0, with the Numerov source (s_(i-1) + 10 s_i + s_(i+1)) / 12, s_i = 2 K_i beta_i e^(-delta i / 2) (uniform grid: 2 h^2 beta_i),
 * in the index variable of the sweep; h_x = <beta|u_x> by the sweep rule on 0..i_s (i_s = the largest node with beta != 0);
 * u = (1 - E_KB h_p) u_h + E_KB h_h u_p.  Both solutions run to max(i_c, i_s) + 1, each rescaled by exact powers of two (u_p with its
 * source), and are combined in one common scale.  u'(r_c) is the fourth-order index derivative of dftatom_log_derivatives less the
 * source term E_KB h_h (s_(i_c+1) - s_(i_c-1)) / 12; int_0^rc u^2 dr is assembled from the running sums of u_h^2, u_h u_p and u_p^2;
 * nodes = sign changes among the non-zero values of u at nodes 1..i_c, and u > 0 at the first of them.  1 - g_i <= 0 at some node
 * 2..max(i_c, i_s) + 1: nodes = -1, NaN.
 * Validation: that of dftatom_log_derivatives (pot, l, r_c, E, V_loc) plus NULL beta with a projector, n_proj < 0, proj outside
 * -1..n_proj-1, E_KB not finite, beta not finite, or i_s > N - 3. */
typedef struct { int pot, proj, l, pad; double E_KB, r_c; } dftatom_kb_ld_channel;                         /* 32 bytes */
int dftatom_kb_log_derivatives(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* V_loc, int n_pot,
                               const double* beta, int n_proj, const dftatom_kb_ld_channel* ch, int n_channels,
                               const double* E, int n_energies, dftatom_logderiv* out, double* r_used);
/* Self-consistent pseudo-atoms: the valence-only atom of semilocal ionic pseudopotentials (e.g. v_ion of dftatom_tm_pseudize), solved
 * in any valence configuration by the SCF of dftatom_solve_batch_config - the transferability test of a pseudopotential: total-energy
 * differences and eigenvalues between configurations against the all-electron atom in the same configurations.
 * Grid (levels, delta, max_r): the logarithmic grid of the SCF (delta = 0, the uniform grid, returns DFTATOM_E_BAD_OPTION).
 * v_ion[n_rows][N] HOST ionic potentials (node 0 ignored).  Atom a = atoms[a]: row[l] the v_ion row of channel l (-1 = no channel),
 * n_ref[l] the all-electron principal number of the channel's reference state (3 for Si 3s), z_val the ionic charge, mixing and method
 * (0 = LDA, 1 = LSDA) as in dftatom_options.  configs[a]: its valence configuration, entries (n, l, spin, occ) with all-electron labels
 * and the occupation rules of dftatom_solve_batch_config; an entry is solved with n - n_ref[l] nodes.
 * Every SCF step runs the all-electron loop in the same order with
 *   V_l,s = V_ion,l + U / r + V_xc,s(rho),  U the Poisson solution of the valence density with boundary value Q = sum occ, V_xc the
 *   VWN LDA (method 0) or LSDA (method 1) of the SCF;
 * every entry is solved in its V_l,s, then the density is built and mixed as in the all-electron SCF.  The stop test, the step caps (100
 * LDA / 150 LSDA), the mixing, the start density (a uniform sphere of Q electrons) and the option "adaptive_mixing" are those of the
 * all-electron SCF.  The energy search brackets [-Z_b^2 - 1, 50], Z_b the smallest integer >= 1 with -Z_b^2 - 1 at least 10 Ha below
 * min over the atom's channels and nodes 1..N-1 of V_ion,l (the margin covers V_xc); its step-0 ladder uses Z_b in place of Z.
 * Reported energies (dftatom_result / dftatom_step):
 *   Eenuc  E_ion = sum occ <u|V_ion,l|u>          Ecoul  E_H            Exc  E_xc
 *   Ekin   sum occ eps - sum occ <u|V_l,s|u>     Etotal sum occ eps - E_H + int rho (eps_xc - v_xc), the all-electron formula; at
 *          convergence Etotal = Ekin + Eenuc + Ecoul + Exc
 *   (<u|f|u> = sum over nodes 1..N-1 of wjac_i u_i^2 f_i with the normalised orbital of the step and the potential built in the step.)
 * dftatom_result.levels[s][k]: n the all-electron label, nodes = n - n_ref[l].  steps, steps_stride and radial as in
 * dftatom_solve_batch_config; the radial export's `v` holds the l-independent screening V_H + V_xc,s per spin (V_l,s = v_ion row + v).
 * The atoms of one call are solved in one group (no stream-group split): a pseudo-atom's records do not depend on the batch.
 * Validation before anything runs on the device (outputs untouched): DFTATOM_E_BAD_OPTION, naming the atom and the entry, for a bad grid or
 * mixing, a method other than 0 / 1, no channel, a row outside -1..n_rows-1, n_ref[l] outside l+1..8, z_val not finite or <= 0, an empty
 * configuration, the occupation ranges and duplicates of dftatom_solve_batch_config, an entry whose l has no channel or with n < n_ref[l],
 * Q outside (0, z_val + 2], V_ion not finite at nodes 1..N-1, or Z_b > 118; DFTATOM_E_ARG for NULL pointers, n_rows or n_atoms < 1 and a
 * too small radial orbital_rows. */
typedef struct { int row[4], n_ref[4]; double z_val, mixing; int method, pad; } dftatom_pseudo_atom;      /* 56 bytes */
int dftatom_solve_pseudo_batch(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* v_ion, int n_rows,
                               const dftatom_pseudo_atom* atoms, const dftatom_config* configs, int n_atoms, dftatom_result* out,
                               dftatom_step* steps, int steps_stride, const dftatom_radial* radial);
/* dftatom_solve_pseudo_batch with nonlinear core corrections: rho_pc[n_pc_rows][N] HOST partial core densities, pc_row[n_atoms] the row
 * of each atom (-1 = none; pc_row = NULL: no atom has one, which is dftatom_solve_pseudo_batch).  An atom with a core uses
 *   V_l,s = V_ion,l + U / r + V_xc,s(rho_a + rho_pc / 2, rho_b + rho_pc / 2)   (LDA: V_xc(rho + rho_pc)),
 *   Exc = int (rho + rho_pc) eps_xc 4 pi r^2 dr,  Etotal = sum occ eps - E_H - sum_s int rho_s v_xc,s 4 pi r^2 dr + Exc;
 * Eenuc, Ecoul and Ekin as before (at convergence Etotal = Ekin + Eenuc + Ecoul + Exc still holds); the radial export's `v` includes the
 * core in V_xc and `rho` stays the valence density.  An atom without a core is solved exactly as by dftatom_solve_pseudo_batch.
 * Validation adds DFTATOM_E_BAD_OPTION, naming the atom or row, for a pc_row outside -1..n_pc_rows-1 (rho_pc = NULL counts as no row)
 * and, when some atom has a core, for a rho_pc row that is not finite or negative at nodes 1..N-1. */
int dftatom_solve_pseudo_batch_core(dftatom_ctx* ctx, int levels, double delta, double max_r, const double* v_ion, int n_rows,
                                    const dftatom_pseudo_atom* atoms, const dftatom_config* configs, int n_atoms, dftatom_result* out,
                                    dftatom_step* steps, int steps_stride, const dftatom_radial* radial, const double* rho_pc,
                                    int n_pc_rows, const int* pc_row);
/* The node radii r[N] (HOST) of the grid (levels, delta, max_r; delta = 0: uniform) as the engine builds and uses them. */
int dftatom_grid_nodes(dftatom_ctx* ctx, int levels, double delta, double max_r, double* r);
/* SolvePoissonNonUniform (PoissonSolver.h:51-81) for n_dens densities rho[n_dens][N] with boundary values (0, Z[k]) (the SCF passes the
 * electron count as a double; Z[k] is converted exactly) */
int dftatom_poisson_solve(dftatom_ctx* ctx, int levels, double delta, double max_r, int n_dens, const int* Z,
                          const double* rho, double* U, int* vcycles_used);
/* One warm Poisson solve of the SCF in increment form for n_dens densities on the grid (levels 8..20, delta, max_r; delta = 0: uniform):
 *     -a dU_{i-1} + dU_i - b dU_{i+1} = psrc_i (rho_i - rho_prev_i) / 2,   a = (1 + delta/2)/2,  b = (1 - delta/2)/2,  dU_0 = dU_{N-1} = 0,
 * then U += dU and rho_prev = rho (psrc_i = r_i 4 pi K_i, the source factor of dftatom_poisson_solve).  rho[n_dens][N]; rho_prev[n_dens][N] and
 * U[n_dens][N] are in / out.  skip (optional, [n_dens]): a density with skip[k] != 0 is left untouched.  solver selects the path the SCF takes:
 *   0  the direct solve (poisson_direct.cu: Thomas algorithm as block scans; 11..20 levels), the SCF's from step "direct_after" on;
 *   1  n_vcycles V-cycles of the warm kernel (poisson_warm.cu; 11..14 levels, delta > 0), the SCF's earlier warm steps there;
 *   2  n_vcycles V-cycles of the cold solvers on the increment (poisson_delta_prepare, poisson_full_kernel or - under the SCF's condition
 *      for a batch of n_dens atoms - the stream-mode solver, poisson_delta_apply), the SCF's warm steps everywhere else.
 * With the launches and arguments of the SCF (the same code); a component entry point for tests.  DFTATOM_E_ARG where the SCF never runs
 * that solver (solver 0 below 11 levels, solver 1 outside 11..14 levels, on the uniform grid or in stream mode, any solver with
 * "poisson_exact", "refine_vcycles" or "floor_stop" set), for NULL pointers and for n_vcycles outside 1..1000 (solvers 1, 2). */
int dftatom_poisson_increment(dftatom_ctx* ctx, int levels, double delta, double max_r, int n_dens, const double* rho, double* rho_prev,
                              double* U, const int* skip, int solver, int n_vcycles);
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
