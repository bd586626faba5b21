// Internal declarations shared by the CUDA translation units of libdftatom_b200.so.
// Data layout in HBM (all FP64, contiguous, index = radial node i, N = 2^L + 1):
//   grid tables  (one set per batch, shared by all atoms):  r, ex=e^{δi}, sqex=e^{δi/2}, b12, c6, k2, simpson-weighted jacobians
//   per (atom,spin): rho[N], atab[N] (a_i = (2 K_i V_i + δ²/4)/12, the potential part of f_i/12), vpot[N]
//   per atom:        rhot[N] (total density; aliases rho of spin 0 for LDA), Poisson hierarchy phi/src (2N-ish each)
//   per orbital:     psi[N], search state
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <string>
#include <vector>
#include "../../include/dftatom_b200.h"

#define DFT_CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { dft::set_error(std::string(#x) + ": " + cudaGetErrorString(e_)); return DFTATOM_E_CUDA; } } while (0)

namespace dft {

void set_error(const std::string& s);

constexpr double kEnergyTol = 1e-12;        // energyErr, DFTAtom.cpp:348
constexpr double kTotalEnergyTol = 1e-11;   // totalEnergyErr, DFTAtom.cpp:349
constexpr double kTopEnergy = 50.0;         // DFTAtom.cpp:499
constexpr double kFarLog = -460.51701859880916;   // ln(1e-200): Numerov.h:195 cut-off
constexpr double kFourPi = 12.566370614359172;

// Grid-only tables (device pointers).  K_i = Rp^2 δ^2 e^{2δ i}  (Numerov.h:85,100; PoissonSolver.h:66-74)
struct GridDev {
    int N, L;
    int uniform;     // 1: the uniform grid of the CalculateUniform* pair (delta == 0): r_i = i h, h = MaxR / (N - 1)   (DFTAtom.cpp:65-67)
    double delta, rp, max_r;
    double h;        // uniform grid: its step (0 on the logarithmic grid)
    double* r;       // r_i = Rp (e^{δ i} - 1)                      (Numerov.h:181-184)
    double* ex;      // e^{δ i}
    double* sqex;    // e^{δ i / 2}                                  (DFTAtom.cpp:42)
    double* b12;     // K_i / (12 r_i^2)   (b12[0] = 0)              centrifugal part of 1 - f/12
    double* c6;      // K_i / 6                                      energy part of 1 - f/12
    double* k2;      // 2 K_i                                        potential part of f
    double* wjac;    // simpson38 weight_i * Rp δ e^{δ i}            (Integral.h:50-73 × jacobian DFTAtom.cpp:47,442)
    double* psrc;    // r_i * 4π K_i  (0 at i=0 and i=N-1)           (PoissonSolver.h:55-74)
    double* inv4pr2; // 1 / (4π r_i^2) (0 at i=0)                    (DFTAtom.cpp:340)
    double* pex;     // 4π Rp²δ² · e^{2δ i} in the reference's own product order (PoissonSolver.h:66-74; uniform grid: h² 4π, :26-40): poisson_exact.cu
    double* coarse_op; // [32*32] dense operator of the Poisson sub-cycle below the 32-node level (poisson.cu), NULL for L < 6
    double* coarse_direct; // pivots of the direct solve of the level-0 system (poisson_direct.cu), NULL unless 11 <= L <= 14
    double* coarse_tri; // table of the exact solve of the 1024-node level (poisson_tri.cuh), NULL unless 11 <= L <= 14
};

// One orbital = one (atom, spin, n, l) level; also the unit of the batched energy search.
struct OrbitalDev {
    int atom, spin, n0, l, occ;
    int want;            // n0 - l = number of nodes (DFTAtom.cpp:497)
    int tab;             // index of the (atom,spin) table row
};

// Search state, one per orbital (device).  Stage A finds both edges of the node-count window
// (LocateInterval, DFTAtom.cpp:566-604), stage B the sign change of y(0) inside it (:513-534).
struct SearchState {
    double up_lo, up_hi;     // bracket of the upper edge (count > want above it)
    double dn_lo, dn_hi;     // bracket of the lower edge (count < want below it)
    double bot, top;         // stage B bracket
    double y0_log2;          // log2|y0| of the last stage-B midpoint (1e15 guard)
    double E;                // result (= bot)
    int stage;               // 0 = A, 1 = B first round (needs sign at bot), 2 = B, 3 = done
    int sgn_bottom;
    int converged;
    int pad;
};

struct AtomDev {
    int Z, method, n_spin, n_steps_max;
    double mixing;
    int orb_begin[2], orb_count[2];
    int n_el[2];
};

struct AtomState {
    double e_old;
    int prev_ok;
    int done;            // 1 once the stop criterion fired or the cap was reached
    int n_steps;
    int status;
    // opt-in adaptive damping (set_option "adaptive_mixing"; beyond the reference, SURVEY 8(f) rank 4): the weight of the OLD density this atom
    // currently mixes with (starts at Options::alpha), the last two changes of Etotal, and a hold-off counter
    double mix, d1, d2;
    int hold, n_raised;
};

struct PoissonLevels {       // offsets of each level inside one density's phi/src block
    int L;
    int off[24];
    int size[24];
    int total;
};
PoissonLevels make_levels(int L);

// ---- launchers (all asynchronous on `st`) ----
struct NumerovLaneArgs {
    const double* atab;   // [n_tabs][N]
    int n_lanes;
    const int* tab; const int* l; const double* E; const int* limit;   // device arrays
    int* y0_sign; double* y0_log2; int* count;
};
void launch_numerov_lanes(const GridDev& g, const NumerovLaneArgs& a, cudaStream_t st);
void launch_numerov_lanes_outward(const GridDev& g, const NumerovLaneArgs& a, cudaStream_t st);     // Numerov.h:204-270

void launch_search_init(const GridDev& g, const AtomDev* atoms, const AtomState* astate, const OrbitalDev* orbs, SearchState* ss,
                        int n_orbs, cudaStream_t st);
void launch_search_round(const GridDev& g, const double* atab, const OrbitalDev* orbs, const AtomState* astate, SearchState* ss,
                         int n_orbs, unsigned long long* work, cudaStream_t st);
void launch_numerov_lanes_fast(const GridDev& g, const NumerovLaneArgs& a, cudaStream_t st);
// n_active_orbs (device, may be NULL) and threshold select between the two search kernels on the device: the serial-in-r
// kernel runs while *n_active_orbs > threshold, the parallel-in-r kernel once *n_active_orbs <= threshold
void launch_search_fused(const GridDev& g, const double* atab, const AtomDev* atoms, const OrbitalDev* orbs, const AtomState* astate,
                         SearchState* ss, int n_orbs, unsigned long long* work, const int* n_active_orbs, int threshold, int warm_start,
                         cudaStream_t st);
void launch_search_seg(const GridDev& g, const double* atab, const AtomDev* atoms, const OrbitalDev* orbs, const AtomState* astate,
                       SearchState* ss, int n_orbs, unsigned long long* work, int segments, const int* n_active_orbs, int threshold,
                       int warm_start, cudaStream_t st);
// lanes through the parallel-in-r sweep: one cluster per 32 lanes sharing (tab, l); segments = 4 x cluster size (<= 32)
void launch_numerov_lanes_seg(const GridDev& g, const NumerovLaneArgs& a, int segments, cudaStream_t st);
// production search (numerov_rows.cu): lanes across the radial grid, 4 trial energies per thread, one CTA of 4 warps per orbital
int launch_search_rows(const GridDev& g, const double* atab, const AtomDev* atoms, const OrbitalDev* orbs, const AtomState* astate,
                        SearchState* ss, int n_orbs, unsigned long long* work, int warm_start, int cfg, int wide_from_step, int step_lo, int step_hi, cudaStream_t st);
// lanes through the same sweep: one CTA per 4 n_groups consecutive lanes (n_groups = 1, 2, 4)
void launch_numerov_lanes_rows(const GridDev& g, const NumerovLaneArgs& a, int n_groups, cudaStream_t st);
int rows_init_device();
void launch_dfma_peak(double* out, int blocks, int threads, int iters, cudaStream_t st);
int search_rounds_needed(int Zmax);

void launch_match(const GridDev& g, const double* atab, const OrbitalDev* orbs, const AtomState* astate, const SearchState* ss,
                  double* psi, int* match_pt, int n_orbs, cudaStream_t st);

void launch_match_seg(const GridDev& g, const double* atab, const OrbitalDev* orbs, const AtomState* astate, const SearchState* ss,
                      double* psi, int* match_pt, int n_orbs, cudaStream_t st);

int launch_match_cta(const GridDev& g, const double* atab, const OrbitalDev* orbs, const AtomState* astate, const SearchState* ss,
                      double* psi, int* match_pt, double* inv_norm, int n_orbs, int win_until_step, int win_nodes, int step_lo, int step_hi, cudaStream_t st);

// potential -> a-table (a_i = 1 - (2K_i V_i + δ²/4)/12), n_tabs rows
void launch_build_atab(const GridDev& g, const double* vpot, double* atab, int n_tabs, cudaStream_t st);

// Poisson
struct PoissonArgs {
    int n_dens;
    const double* rho;      // [n_dens][N] total density, natural node order (or NULL)
    const double* src_nat;  // [n_dens][N] Source_0 in natural node order, used when rho is NULL (or NULL)
    double* u_out;          // [n_dens][N] result U(r) = Phi_0 in natural node order (or NULL)
    long long nat_stride;   // row stride of rho / src_nat / u_out / u0 in doubles (0: N)
    const int* Zbc;         // [n_dens] boundary value at Rmax (may be NULL: use hi_bc)
    double* phi; double* src;   // [n_dens][levels.total] the hierarchy, thread-major node order inside a level (poisson.cu)
    const int* skip;        // optional per-density skip flag (AtomState.done), stride given
    int skip_stride_bytes;
    int max_vcycles; int floor_stop;
    int warm_vcycles;       // > 0: keep Phi_0 of the previous solve as the initial guess and run this many V-cycles (no FMG ramp)
    int n_sm;               // SM count of the context's device (team mode sizing); 0: 148
    int team_G;             // set by the launcher: CTAs per density (team mode, poisson.cu), 1 = off
    unsigned* team_bar;     // [n_dens] scratch for the team barriers (or NULL: no team mode)
    int smem_doubles;       // set by the launcher: doubles per shared-memory array of the coarse levels
    int refine_vcycles;     // > 0: double-double defect correction with this many V-cycles on the error equation
    double* u0;             // [n_dens][N] scratch for the correction (required when refine_vcycles > 0)
    const double* coarse_op; // [32*32] dense operator of the coarse sub-cycle (GridDev.coarse_op) or NULL: run it level by level
    long long* dbg;         // optional [128] cycle counters of CTA 0 (development aid)
    unsigned long long* work;   // optional: += Gauss-Seidel node-updates performed
    int* vcycles_used;      // optional [n_dens]
    double* last_err;       // optional [n_dens]
};
void launch_coarse_op(int L, double delta, double* G, cudaStream_t st);
void launch_poisson_full(const GridDev& g, const PoissonLevels& lv, const PoissonArgs& a, cudaStream_t st);
// U[k][i] = Z[k] u1[i]: the Poisson solve of the SCF's start density from the solution of the Z = 1 problem (engine.cpp: unit_guess)
void launch_scale_unit_potential(int N, int n_dens, int ldU, const double* u1, const int* Z, double* U, cudaStream_t st);
void launch_poisson_vcycles(const PoissonLevels& lv, double delta, int n_dens, double* phi, double* src, double* phi_nat,
                            const double* src_nat, int n_cycles, double* last_err, cudaStream_t st);

// Poisson, stream mode (poisson_stream.cu + poisson_mid_kernel): many densities on a grid that does not fit on chip
enum { kVisitLoadPhi = 1, kVisitProlongIn = 2, kVisitRestrictOut = 4 };
struct StreamVisitArgs {
    double* phi_f; const double* src_f; long long stride_f;   // level l of density k at phi_f + k stride_f (natural node order, 16-byte aligned rows)
    double* phi_c; double* src_c; long long stride_c;         // level l+1
    int n;                  // owned nodes of level l (2^(L-l)); node n is the right boundary
    int slab, HL;           // set by the launcher
    int flags, sweeps;
    double a, bcoef, dc;    // (1 + d_l/2)/2, (1 - d_l/2)/2, d_{l+1}                      (PoissonSolver.cpp:56-57, :150)
    const int* skip; int skip_stride_bytes;                   // optional per-density skip flag (AtomState.done)
};
void launch_stream_visit(const StreamVisitArgs& v, int n_dens, int variant, cudaStream_t st);
int stream_window_nodes(int variant);
void launch_poisson_mid(const PoissonLevels& lv, double delta, int K, int n_dens, double* nat_phi, const double* nat_src, long long nat_stride,
                        double* mid_phi, double* mid_src, int mid_total, const double* coarse_op, const int* skip, int skip_stride_bytes,
                        cudaStream_t st);
// Layout of the scratch block of the stream-mode V-cycle (all offsets in doubles, 4-aligned)
struct StreamPlan {
    int L, K;               // levels; K = the first level run by poisson_mid_kernel (2^mid_levels nodes)
    PoissonLevels lv;
    long long cstride;      // per-density block of the natural-order levels 1..K
    int coff[24];           // offset of level l (1..K) inside that block
    int mid_total;          // per-density block of the owner-major levels K..L-1
    long long off_cphi, off_csrc, off_mphi, off_msrc, total;   // inside the scratch block, for n_dens densities
};
// mid_levels: the levels of up to 2^mid_levels nodes are run by one CTA per density (poisson_mid_kernel); 12 <= mid_levels <= 14
// (the streamed levels must hold at least one 4096-node window), L - mid_levels >= 1
StreamPlan make_stream_plan(int L, int n_dens, int mid_levels = 14);
// n_cycles V-cycles (PoissonSolver.h:155-159) on level-0 arrays phi0/src0 [n_dens][ld0] (device, natural order, ld0 % 2 == 0);
// fuse_tops: the up-visit of cycle k and the down-visit of cycle k+1 of level 0 are one visit with 6 sweeps
void launch_poisson_stream_vcycles(const StreamPlan& sp, double delta, int n_dens, double* phi0, const double* src0, long long ld0,
                                   double* scratch, const double* coarse_op, int n_cycles, int fuse_tops, int variant, cudaStream_t st,
                                   long long* launches);
// SolvePoissonNonUniform (PoissonSolver.h:51-81) in stream mode: FullCycle's full-multigrid ramp + n_v V-cycles, or (warm) n_v
// V-cycles from the previous solution held in U.  Source_0 = psrc * rho is built into src0 when rho is given.
struct StreamSolveArgs {
    int n_dens;
    const double* rho; long long rho_stride; const double* psrc;    // optional: densities [n_dens][rho_stride] and the grid's r 4 pi K table
    double* src0; double* U; long long ld0;                         // level 0: Source_0 and the solution U(r) = Phi_0, rows of ld0 doubles
    const int* Zbc;                                                 // [n_dens] boundary value at Rmax
    double* scratch; const double* coarse_op;
    int n_v, warm, variant;
    const int* skip; int skip_stride_bytes;
};
void launch_poisson_stream_solve(const StreamPlan& sp, double delta, const StreamSolveArgs& a, cudaStream_t st, long long* launches);

// Poisson, bit-reproducible mode (poisson_exact.cu): the reference's FullCycle in its own operation order, U equal bit for bit
struct ExactPoissonArgs {
    int n_dens, L;
    double delta;            // deltaGrid (0: uniform grid)
    const double* rho; long long rho_stride;    // [n_dens][rho_stride] densities, natural node order
    const double* r; const double* pex;         // grid tables (GridDev.r, GridDev.pex)
    const int* Zbc;          // [n_dens] boundary value at Rmax
    double* U; long long ldU;                   // [n_dens][ldU] result
    double* work;            // n_dens * exact_poisson_work_doubles(L) doubles
    const int* skip; int skip_stride_bytes;
    int max_vcycles;         // 100 = the reference (PoissonSolver.h:117)
    int* vcycles_used;       // optional [n_dens]
};
long long exact_poisson_work_doubles(int L);
void launch_poisson_exact(const ExactPoissonArgs& a, cudaStream_t st);

// Poisson, cluster mode (poisson_cluster.cu): warm-started V-cycles for 2049 .. 16385 nodes, one cluster of 8 CTAs per density, the
// hierarchy resident in distributed shared memory
struct ClusterPoissonArgs {
    int n_dens;
    const double* rho; long long rho_stride;    // [n_dens][rho_stride] total densities, natural node order
    double* rho_prev;                           // optional [n_dens][rho_stride], in / out: the density of the previous solve.  Given: increment form - the
                                                // V-cycles solve A dU = -r 4 pi K (rho - rho_prev) from dU = 0 and U += dU (see scf.cu); NULL: they iterate on U
    double* U; long long ldU;                   // [n_dens][ldU] in: previous solution (initial guess), out: U(r)
    const int* Zbc;                             // [n_dens] boundary value at Rmax
    const double* coarse_op;                    // GridDev.coarse_op
    const double* coarse_tri;                   // GridDev.coarse_tri or NULL.  Given: the levels below 2048 nodes are replaced by the exact solve of the
                                                // 1024-node level (poisson_tri.cuh); NULL: they are visited like the reference does, down to the dense operator
    const int* skip; int skip_stride_bytes;
    const int* step; int step_min, step_max;    // optional: the density's SCF step counter (AtomState.n_steps, stride = skip_stride_bytes): it is solved by this launch
                                                // only while step_min <= *step < step_max - two kernels that share the warm solves of one SCF by step index
                                                // (a property of the atom alone: the records stay independent of what else is in the batch)
    int n_vcycles;
    double* scratch; long long scratch_stride;  // poisson_direct.cu above 16385 nodes: n_dens x scratch_stride doubles (>= N - 1 each)
    unsigned long long* work;                   // optional: += Gauss-Seidel node-updates
    int smem_doubles;                           // set by the launcher
    long long* dbg;                             // optional [8 * 32] cycle counters of the first density's CTAs (development aid)
};
bool poisson_cluster_supported(int L, double delta);
void launch_poisson_cluster(const GridDev& g, const ClusterPoissonArgs& a, cudaStream_t st);
int poisson_cluster_init_device();

// Poisson, warm solves in increment form on one SM per density (poisson_warm.cu): the arguments of the cluster mode with rho_prev given;
// gphi / gsrc: scratch of n_dens x gstride doubles each (gstride >= poisson_warm_scratch_doubles(L)), contents irrelevant before and after
bool poisson_warm_supported(int L, double delta);
long long poisson_warm_scratch_doubles(int L);
void launch_poisson_warm(const GridDev& g, const ClusterPoissonArgs& a, double* gphi, double* gsrc, long long gstride, cudaStream_t st);
int poisson_warm_init_device();
// Poisson, warm solves in increment form as one direct (Thomas) solve per density (poisson_direct.cu): the arguments of the cluster mode with rho_prev given
bool poisson_direct_supported(int L);
long long poisson_direct_table_doubles(int L);
void coarse_direct_host(int L, double delta, double* W);      // host-side table builders (once per grid)
void launch_poisson_direct(const GridDev& g, const ClusterPoissonArgs& a, cudaStream_t st);
int poisson_direct_init_device();
void coarse_tri_host(int L, double delta, double* T);

// per-device kernel attributes (opt-in dynamic shared memory): called once per context from dftatom_create under cudaSetDevice
int poisson_init_device();
int stream_init_device();
int match_init_device();

// XC
void launch_vwn(int n, const double* ra, const double* rb, double* va, double* vb, double* vexc, double* edif, cudaStream_t st);
void launch_chachiyo(int n, const double* rho, int improved, double* vexc, double* edif, cudaStream_t st);
void launch_simpson38(double step, const double* v, int n, int n_rows, double* out, cudaStream_t st);
void launch_integrate(int rule, double step, const double* v, int n, int n_rows, double* out, cudaStream_t st);

// SCF pieces (scf.cu)
struct ScfBuffers {
    int n_atoms, n_orbs, n_tabs, N;
    AtomDev* atoms; AtomState* astate; OrbitalDev* orbs; SearchState* ss;
    double* rho;      // [n_tabs][N] per-spin densities
    double* rhot;     // [n_atoms][N] total density
    double* vpot;     // [n_tabs][N]
    double* atab;     // [n_tabs][N]
    double* psi;      // [n_orbs][N]
    int* match_pt;    // [n_orbs]
    double* epart;    // [n_atoms][<= 64 node ranges][5] partial sums of the five energy integrals (potential_energy_kernel)
    int* eticket;     // [n_atoms] arrival counter of its CTAs (zero between launches)
    double* inv_norm; // [n_orbs] 1 / integral u^2 dr of the matched solution in psi
    double* phi; double* src;   // Poisson hierarchy [n_atoms][levels.total]
    double* U;        // [n_atoms][ldU] Hartree U(r) = r V_H, natural node order (output of the Poisson solve)
    int ldU;          // row stride of U (N, or N rounded up to a multiple of 4 when the stream-mode Poisson solver writes it)
    int* Zbc;         // [n_atoms]
    int* tab_of;      // [n_atoms][2] table row of (atom, spin) or -1
    dftatom_step* steps;  // [n_atoms][steps_stride]
    int steps_stride;
    int* n_active;    // device counter of atoms not done
    int run_to_cap;   // != 0: the stop test is recorded in dftatom_step.stop_criterion_met but never ends the SCF
    int adaptive_mixing;  // != 0: per-atom damping is raised when Etotal sloshes with period 2 (scf.cu); 0: the reference's fixed linear mixing
};
// Programmatic dependent launch of the kernels of an SCF step: with g_dft_pdl != 0 (option "use_pdl") a step kernel may be scheduled while
// the kernel before it on the stream drains; every such kernel starts with DFT_PDL_WAIT() - before its first global read and before any
// early exit - which returns once the preceding grid has completed and its writes are visible (a no-op for a normal launch).
extern int g_dft_pdl;
#define DFT_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
template <class... KA, class... A>
inline void launch_step_kernel(void (*k)(KA...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = g_dft_pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, k, static_cast<KA>(args)...);
}

struct ScfLoopPhases { cudaGraphConditionalHandle handle[4]; int n; };      // the WHILE nodes of the SCF loop, one per phase (a range of SCF steps), in order
void launch_scf_loop_condition(const ScfLoopPhases& ph, int phase, int step_first, int step_end, const int* n_active, unsigned long long* iterations, cudaStream_t st);
void launch_gather_last_steps(const ScfBuffers& b, dftatom_step* out, cudaStream_t st);
// increment form of the warm-started Poisson solves (scf.cu): dS = r 4 pi K (rho - rho_prev), dU = 0, rho_prev = rho (dS == NULL: only
// the last); U += dU
void launch_poisson_delta_prepare(const GridDev& g, int n_dens, long long ld, const double* rho, double* rho_prev, double* dS, double* dU,
                                  const int* skip, int skip_stride_bytes, cudaStream_t st);
void launch_poisson_delta_apply(const GridDev& g, int n_dens, long long ld, double* U, const double* dU, const int* skip, int skip_stride_bytes,
                                cudaStream_t st);
void launch_initial_density(const GridDev& g, const ScfBuffers& b, cudaStream_t st);
void launch_orbital_norms(const GridDev& g, const ScfBuffers& b, cudaStream_t st);
void launch_density_update(const GridDev& g, const ScfBuffers& b, cudaStream_t st);
void launch_potential_energy(const GridDev& g, const PoissonLevels& lv, const ScfBuffers& b, int first, cudaStream_t st);

// export of the radial state (radial.cu): part / ticket: radial_part_doubles(N, rows) doubles / rows ints (tickets zero before the launch)
long long radial_part_doubles(int N, int n_rows);
void launch_radial_orbitals(const GridDev& g, const double* src, const double* inv_norm, int from_scf, int n_rows, double* u_out, double* moments,
                            double* part, int* ticket, cudaStream_t st);
void launch_radial_fields(const GridDev& g, const ScfBuffers& b, double* rho_out, double* v_out, double* vh_out, double* atom_moments,
                          double* part, int* ticket, cudaStream_t st);

// host rules (aufbau.cpp)
int aufbau(int Z, dftatom_level* out, int max_out);
int split_spin(int Z, dftatom_level* a, int* na, dftatom_level* b, int* nb, int* ea, int* eb);
double estimate_cost(int Z, int method);
int partition_atoms(const int* Z, const int* method, int n, int n_ranks, int* rank_of);

}  // namespace dft
