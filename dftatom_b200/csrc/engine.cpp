// Host side of libdftatom_b200.so: context, grid tables, device buffers, the SCF launch sequence and the C ABI
// declared in include/dftatom_b200.h.  The host only enqueues kernels; densities, potentials, the energy search
// state, mixing and the stop test live on the device (north_star: no per-step host round trip).
#include "internal.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <numeric>
#include <thread>
#include <chrono>
#include <nvtx3/nvToolsExt.h>

namespace dft {

static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }
int g_dft_pdl = 0;         // internal.h: launch_step_kernel (set from the option "use_pdl" when a solve starts)

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); return DFTATOM_E_CUDA; }
        cap = bytes;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() { return static_cast<T*>(p); }
};

struct GridKey {
    int L; double delta, max_r;
    bool operator<(const GridKey& o) const { return std::tie(L, delta, max_r) < std::tie(o.L, o.delta, o.max_r); }
};

struct GridEntry {
    GridDev dev; DevBuf mem;
    std::vector<double> r;                      // the node radii dev.r holds, as uploaded (host checks of radii round to these nodes)
    DevBuf u_unit; bool u_unit_ok = false;      // U of the SCF's start density for Z = 1 (solve_group: unit_guess), [N] doubles + one int (= 1)
};

// CUDA events of one call, destroyed on every return path
struct EventPool {
    std::vector<cudaEvent_t> all;
    bool ok = true;
    cudaEvent_t make(bool timing)
    {
        cudaEvent_t e = nullptr;
        if (cudaEventCreateWithFlags(&e, timing ? cudaEventDefault : cudaEventDisableTiming) != cudaSuccess) { ok = false; return nullptr; }
        all.push_back(e);
        return e;
    }
    ~EventPool() { for (cudaEvent_t e : all) cudaEventDestroy(e); }
};

}  // namespace dft

using namespace dft;

// Tuning knobs of a context, set through dftatom_set_option (documented in include/dftatom_b200.h).  One struct so that the
// child context of stream_groups = 2 inherits ALL of them by assignment.
struct Knobs {
    int max_vcycles = 8;
    int floor_stop = 0;
    int refine_vcycles = 0;
    int warm_vcycles = 7;      // Poisson warm start from SCF step warm_after on: V-cycles per solve (0 = always the full cycle)
    int warm_after = 1;
    int team_poisson = 1;      // large grids, few atoms: several CTAs per density (poisson.cu, team mode)
    int r_segments = -1;       // radial segments per orbital of the parallel-in-r search; -1 = auto (16 up to 16385 nodes, 32 above), 0 / 1 = serial-in-r search only
    int seg_threshold = 2400;  // the parallel-in-r search runs once at most this many orbitals are still active; above it (>= 4 warps per
                               // FP64 pipe) the serial-in-r kernel, one warp per orbital, is throughput-bound with 8 instead of 11 FP64
                               // instructions per (lane, node) and wins (8 x C3 in one batch: 1135 against 975 atoms/s)
    int segments(int N) const { return r_segments < 0 ? (N <= 16385 ? 16 : 32) : r_segments; }
    int profile = 0;
    int search_mode = 0;
    int search_kernel = 0;     // search_mode 0 on the logarithmic grid: 0 = lanes across the radial grid, 4 trial energies per thread, one CTA per orbital
                               // (numerov_rows.cu, production); 1 = lanes across 32 trial energies, cluster per orbital (numerov_seg.cu / numerov_fast.cu)
    int rows_wide_from_step = 32;   // numerov_rows.cu: from this SCF step on an atom's orbitals are searched by the 8-warp shape (0 = never)
    int rows_cfg = 0x111;      // numerov_rows.cu: energy groups of 4 per round - first ladder of a warm start (bits 0-3), later ladders (4-7), uniform rounds (8-11)
    int match_mode = 0;
    int match_win_until_step = 32;  // > 0 (grids that fit one window of the matched-solution kernel): up to this SCF step the orbitals are solved in windows of
    int match_win_nodes = 8192;     // match_win_nodes nodes (several CTAs per SM), afterwards in one window (numerov_match.cu)
    int warm_start = 1;
    int stream_variant = 0;    // window shape of the stream-mode Poisson visits (poisson_stream.cu)
    int stream_poisson = 1;    // grids above 16385 nodes: level visits streamed over all densities (poisson_stream.cu) instead of one CTA / team per density
    int stream_min_dens = 4;   // ... when the batch has at least this many densities (below, the team of CTAs per density is faster)
    int stream_mid_levels = 11; // stream mode: levels of up to 2^this nodes are run by one CTA per density, the larger ones by slab windows
    int stream_min_levels = 15; // stream mode from this many levels on (at 14 levels one CTA per density is as fast: measured 57.6 against 58.5 ms on C3)
    int poisson_exact = 0;     // 1: bit-reproducible Poisson solve (poisson_exact.cu): the reference's FullCycle in its own operation order, 100 V-cycles
    int run_to_cap = 0;        // 1: the stop test (DFTAtom.cpp:474) is evaluated and recorded but never ends the SCF (trajectory parity beyond the stop step)
    int direct_poisson = 1;    // warm solves in increment form on 2049 .. 16385 nodes: the level-0 system solved directly (Thomas algorithm as block scans,
                               // poisson_direct.cu) instead of 7 V-cycles by one CTA per density (poisson_warm.cu)
    int direct_after = 4;      // ... from this SCF step on (earlier warm steps: the V-cycle kernel)
    int delta_poisson = 1;     // warm-started Poisson solves in increment form (A dU = -dS, U += dU: scf.cu) - keeps consecutive SCF steps free of the
                               // rounding-floor noise of a plain FP64 multigrid solve; 0 = iterate on U itself
    int adaptive_mixing = 0;   // opt-in: per-atom damping raised when Etotal sloshes with period 2 (beyond the reference; default: its fixed linear mixing)
    int step_cap = 0;          // > 0: lower the SCF step cap (100 LDA / 150 LSDA, DFTAtom.cpp:396,908) to this many steps (tests: with run_to_cap, run exactly as long as the reference did)
    int use_graph = 1;         // SCF steps are replayed from a captured CUDA graph (one graph launch per step) instead of 5+ kernel launches
    int unit_guess = 1;        // the Poisson solve of the SCF's start density (a uniform sphere of Z electrons: linear in Z) is done once per grid for Z = 1
                               // and scaled per atom, instead of one cold multigrid solve per atom and call (grids up to 16385 nodes)
    int search_predict = 1;    // rows search: first ladders from what the first SCF steps are known to do (hydrogenic levels of the initial uniform-sphere
                               // potential at step 0, one-sided ladder at step 1, default decay ratio at step 2, miss scaled with the shifts later)
    int use_pdl = 1;           // the kernels of an SCF step are launched with programmatic stream serialization (internal.h: launch_step_kernel)
    int graph_phases = 1;      // the graph loop is a chain of WHILE nodes, one per range of SCF steps between the step indices at which a kernel shape changes
                               // (rows_wide_from_step, match_win_until_step): each body holds only the shapes of its range.  0: one WHILE node, every shape in it
};

struct dftatom_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::map<GridKey, GridEntry> grids;
    Knobs k;                        // tuning knobs (dftatom_set_option); copied as a whole to the child context
    int segments(int N) const { return k.segments(N); }
    int stream_groups = 4;     // a batch of >= 32 atoms (grids up to 16385 nodes) is dealt into this many groups that run their SCF chains concurrently on
                               // separate streams: one group's Poisson solves (one SM per density) overlap another's search; per-atom records are unchanged
    dftatom_ctx* child = nullptr;   // context (stream + buffers) of the second group
    int n_sm = 148;
    DevBuf stream_src0, stream_scratch, exact_work, last_steps, rho_prev, d_src, d_u;
    dftatom_step* h_last = nullptr; size_t h_last_cap = 0;      // pinned staging of the result records
    DevBuf stream_G; int stream_G_levels = 0; double stream_G_delta = 0.;   // dense coarse operator of the stream-mode V-cycle
    dftatom_kernel_profile prof[DFTATOM_K_COUNT] = {};
    // reusable buffers
    DevBuf atoms, astate, orbs, ss, rho, rhot, vpot, atab, psi, match_pt, inv_norm, epart, eticket, team_bar, phi, src, u0, ubuf, zbc, tab_of, steps, n_active;
    DevBuf scratch[8];
    DevBuf radial, radial_part, radial_ticket;     // export of the radial state (dftatom_solve_batch_radial): staging, partial sums, tickets
    DevBuf pseudo_atoms, pseudo_v;                 // dftatom_solve_pseudo_batch: per-atom channel rows, the ionic potentials
    DevBuf pseudo_pc, pseudo_pc_row;               // dftatom_solve_pseudo_batch_core: partial core rows, the row of each atom
    int* h_active = nullptr;       // pinned
    char* h_up = nullptr; size_t h_up_cap = 0, h_up_used = 0;      // pinned staging of the descriptor uploads of one solve (reset at its start)
    // timing of the last solve
    double last_ms = 0.;
    long long last_launches = 0;
    long long last_graph_iterations = 0;                    // SCF steps the last solve ran inside the CUDA-graph while node (0: host-driven loop)
    long long last_d2h_bytes = 0, last_h2d_bytes = 0;      // bytes the last solve_batch moved between host and device
};

namespace dft {

static int get_grid(dftatom_ctx* c, int L, double delta, double max_r, GridDev** out, GridEntry** entry_out = nullptr)
{
    // one place for the grid arguments of every entry point: 1 <= levels <= 22 (PoissonLevels holds 24, shifts stay defined), finite
    // delta >= 0 (0 = uniform grid) and finite max_r > 0 (a NaN would also break the ordering of the grid cache)
    if (L < 1 || L > 22 || !(delta >= 0.) || !std::isfinite(delta) || !(max_r > 0.) || !std::isfinite(max_r)) {
        set_error("bad grid: need 1 <= levels <= 22, finite delta >= 0, finite max_r > 0");
        return DFTATOM_E_BAD_OPTION;
    }
    const GridKey key{ L, delta, max_r };
    auto it = c->grids.find(key);
    if (it != c->grids.end()) { *out = &it->second.dev; if (entry_out) *entry_out = &it->second; return 0; }
    const int N = (1 << L) + 1;
    // host tables with the same libm the CPU reference uses (exp), uploaded once per grid
    const int n_tab = 10;
    std::vector<double> h((size_t)n_tab * N);
    double* r = &h[0]; double* ex = &h[(size_t)N]; double* sqex = &h[(size_t)2 * N]; double* b12 = &h[(size_t)3 * N];
    double* c6 = &h[(size_t)4 * N]; double* k2 = &h[(size_t)5 * N]; double* wjac = &h[(size_t)6 * N];
    double* psrc = &h[(size_t)7 * N]; double* inv4pr2 = &h[(size_t)8 * N]; double* pex = &h[(size_t)9 * N];
    // delta == 0 selects the UNIFORM grid of the CalculateUniform* pair (DFTAtom.cpp:65-67: h = MaxR / (N - 1), r_i = i h): the same
    // tables with e^{delta i} = 1 and K_i = h^2 (Numerov.h:26-31 times h^2; PoissonSolver.h:22-43).  Only the component entry points
    // accept it so far (dftatom_poisson_solve); dftatom_solve_batch validates delta in (0, 1].
    const bool uniform = delta == 0.;
    const double h_uni = max_r / (double)(N - 1);
    const double rp = uniform ? 0. : max_r / (std::exp((double)(N - 1) * delta) - 1.);      // DFTAtom.cpp:356
    const double rp2d2 = rp * rp * (delta * delta);
    for (int i = 0; i < N; ++i) {
        ex[i] = std::exp((double)i * delta);
        r[i] = uniform ? (0. * (double)(N - 1 - i) + max_r * (double)i) / (double)(N - 1) : rp * (ex[i] - 1.);   // PoissonSolver.cpp:199-209 / Numerov.h:181-184
        sqex[i] = std::exp((double)i * delta * 0.5);                         // DFTAtom.cpp:42
        const double K = uniform ? h_uni * h_uni : rp2d2 * std::exp((double)i * (2. * delta));        // Numerov.h:100
        b12[i] = i ? K / (12. * r[i] * r[i]) : 0.;
        c6[i] = K / 6.;
        k2[i] = 2. * K;
        const double w = (i == 0 || i == N - 1) ? 1. : ((i % 3 == 0) ? 2. : 3.);   // Integral.h:50-73
        wjac[i] = 0.375 * w * (uniform ? h_uni : rp * delta * ex[i]);        // jacobian DFTAtom.cpp:47,442 (uniform: the step h, :182)
        psrc[i] = (i == 0 || i == N - 1) ? 0. : r[i] * (kFourPi * K);        // PoissonSolver.h:55-74
        inv4pr2[i] = i ? 1. / (kFourPi * r[i] * r[i]) : 0.;                  // DFTAtom.cpp:340
    }
    {   // the source factor of the bit-reproducible Poisson mode, in the reference's own product order
        const double four_pi = 4. * M_PI;                                   // fourM_PI, PoissonSolver.h:12
        if (uniform) {
            const double dlt = r[1] - r[0];                                 // PoissonSolver.h:26-27
            const double d2f = (dlt * dlt) * four_pi;                       // :39
            for (int i = 0; i < N; ++i) pex[i] = d2f;
        } else {
            const double rp_p = max_r / (std::exp(((double)N - 1.) * delta) - 1.);      // PoissonSolver.h:65
            const double f = four_pi * (rp_p * rp_p * (delta * delta));     // :66-70
            const double twodelta = 2. * delta;
            for (int i = 0; i < N; ++i) pex[i] = f * std::exp(i * twodelta);            // :74
        }
    }
    GridEntry& e = c->grids[key];
    e.r.assign(r, r + N);
    int rc = e.mem.ensure((h.size() + 32 * 32 + 3 * 1024 + (size_t)poisson_direct_table_doubles(L)) * sizeof(double));
    if (rc) { c->grids.erase(key); return rc; }
    DFT_CHECK(cudaMemcpyAsync(e.mem.p, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    DFT_CHECK(cudaStreamSynchronize(c->stream));
    double* d = e.mem.as<double>();
    e.dev.N = N; e.dev.L = L; e.dev.delta = delta; e.dev.rp = rp; e.dev.max_r = max_r;
    e.dev.uniform = uniform ? 1 : 0; e.dev.h = uniform ? h_uni : 0.;
    e.dev.r = d; e.dev.ex = d + (size_t)N; e.dev.sqex = d + (size_t)2 * N; e.dev.b12 = d + (size_t)3 * N;
    e.dev.c6 = d + (size_t)4 * N; e.dev.k2 = d + (size_t)5 * N; e.dev.wjac = d + (size_t)6 * N;
    e.dev.psrc = d + (size_t)7 * N; e.dev.inv4pr2 = d + (size_t)8 * N; e.dev.pex = d + (size_t)9 * N;
    e.dev.coarse_op = nullptr; e.dev.coarse_tri = nullptr; e.dev.coarse_direct = nullptr;
    if (L >= 6) {
        e.dev.coarse_op = d + (size_t)n_tab * N;
        launch_coarse_op(L, delta, e.dev.coarse_op, c->stream);
        std::vector<double> tab(3 * 1024 + (size_t)poisson_direct_table_doubles(L));      // pivot tables of the exact solves: dependent chains, built here
        if (L >= 11 && L <= 14) {
            e.dev.coarse_tri = d + (size_t)n_tab * N + 32 * 32;
            coarse_tri_host(L, delta, tab.data());
        }
        if (poisson_direct_supported(L)) {
            e.dev.coarse_direct = d + (size_t)n_tab * N + 32 * 32 + 3 * 1024;
            coarse_direct_host(L, delta, tab.data() + 3 * 1024);
        }
        DFT_CHECK(cudaMemcpyAsync(d + (size_t)n_tab * N + 32 * 32, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        DFT_CHECK(cudaStreamSynchronize(c->stream));
    }
    *out = &e.dev;
    if (entry_out) *entry_out = &e;
    return 0;
}

static int validate(const dftatom_options& o)
{   // ranges of the reference's dialog validators, OptionsFrame.cpp:46,152-173 (levels: the class itself accepts any >= 1)
    if (o.Z < 1 || o.Z > 118) { set_error("Z must be in 1..118"); return DFTATOM_E_BAD_OPTION; }
    // the dialog offers 10..20; below 8 levels (257 nodes) 1 - f/12 turns negative over much of the grid and the reference's own
    // sweeps stop meaning anything (measured: Ne at 65 nodes, 42 Ha between two evaluation orders of the same recurrence)
    if (o.levels < 8 || o.levels > 20) { set_error("levels must be in 8..20"); return DFTATOM_E_BAD_OPTION; }
    if (!(o.max_r >= 1. && o.max_r <= 90.)) { set_error("max_r must be in 1..90"); return DFTATOM_E_BAD_OPTION; }
    if (o.method < 0 || o.method > 3) { set_error("method must be 0 (LDA), 1 (LSDA), 2 (LDA, uniform grid) or 3 (LSDA, uniform grid)"); return DFTATOM_E_BAD_OPTION; }
    if (o.method < 2 && !(o.delta > 0. && o.delta <= 1.)) { set_error("delta must be in (0,1]"); return DFTATOM_E_BAD_OPTION; }      // unused on the uniform grid
    if (!(o.mixing >= 0. && o.mixing <= 1.)) { set_error("mixing must be in [0,1]"); return DFTATOM_E_BAD_OPTION; }
    return 0;
}

// ---- argument checks shared by the entry points ----

// the message prefix "fn: what k: "
static std::string where(const char* fn, const char* what, long long k)
{
    return std::string(fn) + ": " + what + " " + std::to_string(k) + ": ";
}

// the first node in 1..N-1 of row[N] that is not finite (or, with `negative`, also below 0); 0 if there is none
static int bad_node(const double* row, int N, bool negative = false)
{
    for (int i = 1; i < N; ++i)
        if (!std::isfinite(row[i]) || (negative && row[i] < 0.)) return i;
    return 0;
}

// the node used for a radius r_2 <= r_c <= r_(N-2): the nearest one, ties to the inner one
static int nearest_node(const std::vector<double>& r, double r_c)
{
    const int N = (int)r.size();
    const int hi = (int)(std::lower_bound(r.begin() + 2, r.begin() + (N - 1), r_c) - r.begin());      // first node >= r_c, 2..N-2
    return (hi > 2 && r_c - r[hi - 1] <= r[hi] - r_c) ? hi - 1 : hi;
}

// the node of the radius `name` = x, which must lie in [r_k, r_(N-k)] (k >= 2); -1 with the error set (prefix `at`) if it does not
static int radius_node(const std::vector<double>& r, double x, int k, const std::string& at, const char* name)
{
    const int N = (int)r.size();
    if (!(x >= r[k] && x <= r[N - k])) {
        char b[160];
        std::snprintf(b, sizeof b, "%s = %.17g outside [r_%d, r_(N-%d)] = [%.17g, %.17g]", name, x, k, k, r[k], r[N - k]);
        set_error(at + b);
        return -1;
    }
    return nearest_node(r, x);
}

// the bottom -Z_b^2 - 1 of the energy search's bracket on a potential with minimum vmin: the smallest Z_b in 1..118 with -Z_b^2 - 1 at
// least `margin` below vmin; 0 if there is none
static int bracket_z(double vmin, double margin)
{
    for (int z = 1; z <= 118; ++z)
        if (-(double)z * z - 1. <= vmin - margin) return z;
    return 0;
}

// one warp per (channel, block of eb energies), dealt longest sweep first (stable: equal costs keep channel order): the item
// channel * eb + block of every warp
static std::vector<int> warp_order(const std::vector<long long>& cost, int eb)
{
    std::vector<int> order(cost.size()), item;
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    for (int q : order)
        for (int b = 0; b < eb; ++b) item.push_back(q * eb + b);
    return item;
}

// the radial export of a whole batch: atom a goes to index a of the caller's arrays and its orb_rows[a] orbitals to the rows after those
// of atoms 0..a-1; radial.orbital_rows must hold them all
static int batch_rows(const dftatom_radial& radial, const std::vector<long long>& orb_rows, std::vector<int>& atom, std::vector<long long>& row)
{
    long long rows = 0;
    for (size_t a = 0; a < orb_rows.size(); ++a) { atom.push_back((int)a); row.push_back(rows); rows += orb_rows[a]; }
    if ((radial.orbitals || radial.moments) && radial.orbital_rows < rows) {
        set_error("dftatom_radial.orbital_rows is " + std::to_string(radial.orbital_rows) + ", the batch has " + std::to_string(rows) + " orbitals");
        return DFTATOM_E_ARG;
    }
    return 0;
}

// descriptor upload through the context's pinned arena: truly asynchronous (a copy from pageable memory is staged and synchronised by the
// driver - five of those per group, from four host threads, were ~1 ms of every sweep)
template <class T> static int upload(dftatom_ctx* c, DevBuf& b, const std::vector<T>& h)
{
    int rc = b.ensure(std::max<size_t>(h.size(), 1) * sizeof(T));
    if (rc) return rc;
    if (h.empty()) return 0;
    const size_t bytes = h.size() * sizeof(T), at = (c->h_up_used + 63) & ~(size_t)63;
    if (at + bytes <= c->h_up_cap) {
        std::memcpy(c->h_up + at, h.data(), bytes);
        c->h_up_used = at + bytes;
        DFT_CHECK(cudaMemcpyAsync(b.p, c->h_up + at, bytes, cudaMemcpyHostToDevice, c->stream));
    } else {
        DFT_CHECK(cudaMemcpyAsync(b.p, h.data(), bytes, cudaMemcpyHostToDevice, c->stream));        // (arena too small for this batch: staged copy)
    }
    return 0;
}
// called at the start of a solve: the arena is free again (the previous solve has synchronised its stream); grown to what that solve needed
static int upload_arena_reset(dftatom_ctx* c, size_t want_bytes)
{
    c->h_up_used = 0;
    if (want_bytes > c->h_up_cap) {
        if (c->h_up) cudaFreeHost(c->h_up);
        c->h_up = nullptr; c->h_up_cap = 0;
        const size_t cap = std::max<size_t>(want_bytes * 2, (size_t)1 << 16);
        DFT_CHECK(cudaMallocHost((void**)&c->h_up, cap));
        c->h_up_cap = cap;
    }
    return 0;
}

}  // namespace dft

extern "C" {

const char* dftatom_last_error(void) { return g_err.c_str(); }
const char* dftatom_version(void) { return "dftatom_b200 0.1 (sm_100a)"; }

int dftatom_create(dftatom_ctx** out, int device)
{
    if (!out) return DFTATOM_E_ARG;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        set_error("no CUDA device: dftatom_b200 has no CPU fallback");
        return DFTATOM_E_NO_DEVICE;
    }
    if (device < 0 || device >= n) { set_error("bad device index"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(device));
    dftatom_ctx* c = new dftatom_ctx;
    c->device = device;
    DFT_CHECK(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device));
    // opt-in dynamic shared memory is per-device state: set it here, for this context's device (not cached process-wide)
    int rc_attr;
    if ((rc_attr = poisson_init_device()) || (rc_attr = stream_init_device()) || (rc_attr = match_init_device()) || (rc_attr = rows_init_device()) || (rc_attr = poisson_warm_init_device()) || (rc_attr = poisson_direct_init_device())) { delete c; return rc_attr; }
    DFT_CHECK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    DFT_CHECK(cudaMallocHost((void**)&c->h_active, sizeof(int) * 256));
    *out = c;
    // DFTATOM_OPTIONS="key=value key=value ...": options applied to every new context (profiling aid: e.g. "use_graph=0 stream_groups=1" for a
    // kernel-by-kernel launch list under ncu); an unknown key is an error
    if (const char* env = getenv("DFTATOM_OPTIONS")) {
        std::string e(env);
        size_t pos = 0;
        while (pos < e.size()) {
            size_t end = e.find_first_of(" ,;", pos);
            if (end == std::string::npos) end = e.size();
            const std::string kv = e.substr(pos, end - pos);
            pos = end + 1;
            if (kv.empty()) continue;
            const size_t eq = kv.find('=');
            if (eq == std::string::npos) { set_error("DFTATOM_OPTIONS: expected key=value, got " + kv); dftatom_destroy(c); *out = nullptr; return DFTATOM_E_ARG; }
            const int rc_o = dftatom_set_option(c, kv.substr(0, eq).c_str(), atof(kv.substr(eq + 1).c_str()));
            if (rc_o) { dftatom_destroy(c); *out = nullptr; return rc_o; }
        }
    }
    return 0;
}

void dftatom_destroy(dftatom_ctx* c)
{
    if (!c) return;
    if (c->child) { dftatom_destroy(c->child); c->child = nullptr; }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto& kv : c->grids) kv.second.mem.release();
    DevBuf* all[] = { &c->atoms, &c->astate, &c->orbs, &c->ss, &c->rho, &c->rhot, &c->vpot, &c->atab, &c->psi, &c->match_pt, &c->inv_norm, &c->epart, &c->eticket, &c->team_bar,
                      &c->phi, &c->src, &c->u0, &c->ubuf, &c->zbc, &c->tab_of, &c->steps, &c->n_active };
    for (DevBuf* b : all) b->release();
    for (DevBuf& b : c->scratch) b.release();
    c->radial.release(); c->radial_part.release(); c->radial_ticket.release();
    c->pseudo_atoms.release(); c->pseudo_v.release(); c->pseudo_pc.release(); c->pseudo_pc_row.release();
    c->stream_G.release(); c->stream_src0.release(); c->stream_scratch.release(); c->exact_work.release(); c->last_steps.release(); c->rho_prev.release(); c->d_src.release(); c->d_u.release();
    if (c->h_active) cudaFreeHost(c->h_active);
    if (c->h_up) cudaFreeHost(c->h_up);
    if (c->h_last) cudaFreeHost(c->h_last);
    cudaStreamDestroy(c->stream);
    delete c;
}

int dftatom_set_option(dftatom_ctx* c, const char* key, double value)
{
    if (!c || !key) return DFTATOM_E_ARG;
    const std::string k(key);
    if (k == "max_vcycles") c->k.max_vcycles = std::max(1, (int)value);
    else if (k == "vcycle_floor_stop") c->k.floor_stop = value != 0.;
    else if (k == "refine_vcycles") c->k.refine_vcycles = std::max(0, (int)value);
    else if (k == "warm_vcycles") c->k.warm_vcycles = std::max(0, (int)value);
    else if (k == "warm_after") c->k.warm_after = std::max(0, (int)value);
    else if (k == "team_poisson") c->k.team_poisson = value != 0.;
    else if (k == "r_segments") c->k.r_segments = (int)value;
    else if (k == "seg_threshold") c->k.seg_threshold = (int)value;
    else if (k == "profile") c->k.profile = value != 0.;
    else if (k == "search_mode") c->k.search_mode = (int)value;
    else if (k == "search_kernel") c->k.search_kernel = (int)value != 0;
    else if (k == "rows_wide_from_step") c->k.rows_wide_from_step = std::max(0, (int)value);
    else if (k == "rows_cfg") {
        const int v = (int)value;
        for (int sft = 0; sft < 12; sft += 4) { const int ng = (v >> sft) & 15; if (ng != 1 && ng != 2 && ng != 4) { set_error("rows_cfg: every field must be 1, 2 or 4"); return DFTATOM_E_ARG; } }
        c->k.rows_cfg = v & 0xfff;
    }
    else if (k == "match_mode") c->k.match_mode = (int)value;
    else if (k == "match_win_until_step") c->k.match_win_until_step = std::max(0, (int)value);
    else if (k == "match_win_nodes") c->k.match_win_nodes = std::max(1024, (int)value);
    else if (k == "warm_start") c->k.warm_start = value != 0.;
    else if (k == "stream_groups") c->stream_groups = std::min(8, std::max(1, (int)value));
    else if (k == "stream_poisson") c->k.stream_poisson = value != 0.;
    else if (k == "stream_min_dens") c->k.stream_min_dens = std::max(1, (int)value);
    else if (k == "stream_mid_levels") c->k.stream_mid_levels = std::min(14, std::max(11, (int)value));
    else if (k == "stream_min_levels") c->k.stream_min_levels = std::min(23, std::max(13, (int)value));
    else if (k == "stream_variant") c->k.stream_variant = std::min(2, std::max(0, (int)value));
    else if (k == "poisson_exact") c->k.poisson_exact = value != 0.;
    else if (k == "direct_after") c->k.direct_after = std::max(0, (int)value);
    else if (k == "direct_poisson") c->k.direct_poisson = value != 0.;
    else if (k == "delta_poisson") c->k.delta_poisson = value != 0.;
    else if (k == "adaptive_mixing") c->k.adaptive_mixing = value != 0.;
    else if (k == "step_cap") c->k.step_cap = std::max(0, (int)value);
    else if (k == "run_to_cap") c->k.run_to_cap = value != 0.;
    else if (k == "use_graph") c->k.use_graph = value != 0.;
    else if (k == "graph_phases") c->k.graph_phases = value != 0.;
    else if (k == "use_pdl") c->k.use_pdl = value != 0.;
    else if (k == "search_predict") c->k.search_predict = value != 0.;
    else if (k == "unit_guess") c->k.unit_guess = value != 0.;
    else { set_error("unknown option " + k); return DFTATOM_E_ARG; }
    return 0;
}

int dftatom_aufbau(int Z, dftatom_level* out, int max_out) { return dft::aufbau(Z, out, max_out); }
int dftatom_config_aufbau(int Z, int method, double charge, dftatom_config* out) { return dft::config_aufbau(Z, method, charge, out); }
int dftatom_split_spin(int Z, dftatom_level* a, int* na, dftatom_level* b, int* nb, int* ea, int* eb)
{
    return dft::split_spin(Z, a, na, b, nb, ea, eb);
}
int dftatom_n_nodes(int levels) { return (1 << levels) + 1; }
double dftatom_estimate_cost(int Z, int method) { return dft::estimate_cost(Z, method); }
int dftatom_partition(const int* Z, const int* method, int n_atoms, int n_ranks, int* rank_of) { return dft::partition_atoms(Z, method, n_atoms, n_ranks, rank_of); }

int dftatom_last_timing(dftatom_ctx* c, double* ms, long long* launches)
{
    if (!c) return DFTATOM_E_ARG;
    if (ms) *ms = c->last_ms;
    if (launches) *launches = c->last_launches;
    return 0;
}

int dftatom_last_graph_iterations(dftatom_ctx* c, long long* iterations)
{
    if (!c || !iterations) return DFTATOM_E_ARG;
    *iterations = c->last_graph_iterations;
    return 0;
}

int dftatom_last_transfer(dftatom_ctx* c, long long* h2d_bytes, long long* d2h_bytes)
{
    if (!c) return DFTATOM_E_ARG;
    if (h2d_bytes) *h2d_bytes = c->last_h2d_bytes;
    if (d2h_bytes) *d2h_bytes = c->last_d2h_bytes;
    return 0;
}

int dftatom_last_profile(dftatom_ctx* c, dftatom_kernel_profile* out)
{
    if (!c || !out) return DFTATOM_E_ARG;
    for (int k = 0; k < DFTATOM_K_COUNT; ++k) out[k] = c->prof[k];
    return 0;
}

int dftatom_measure_fp64_peak(dftatom_ctx* c, double* tflops)
{
    if (!c || !tflops) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int blocks = 148 * 8, threads = 256, iters = 1 << 15;
    int rc = c->scratch[0].ensure(sizeof(double) * (size_t)blocks * threads);
    if (rc) return rc;
    cudaEvent_t a, b;
    DFT_CHECK(cudaEventCreate(&a)); DFT_CHECK(cudaEventCreate(&b));
    double best = 0.;
    for (int rep = 0; rep < 6; ++rep) {
        DFT_CHECK(cudaEventRecord(a, st));
        launch_dfma_peak(c->scratch[0].as<double>(), blocks, threads, iters, st);
        DFT_CHECK(cudaEventRecord(b, st));
        DFT_CHECK(cudaEventSynchronize(b));
        float ms = 0.f;
        DFT_CHECK(cudaEventElapsedTime(&ms, a, b));
        const double fl = 2. * 8. * (double)iters * blocks * threads;
        if (rep >= 1) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    *tflops = best;
    return 0;
}

// Where the radial arrays of the atoms of one group go in the caller's arrays: per local atom its index in the caller's batch and its
// first orbital row (a group of a stream-group split holds a permuted subset of the batch)
struct RadialDest {
    const dftatom_radial* rad;
    const int* atom;
    const long long* row;
    bool copy_r;               // this group copies the grid nodes (once per call)
};

// The radial state of the group's atoms: packed into the staging buffer by radial.cu, then one copy per contiguous block of the
// caller's arrays (a run of atoms whose destinations are consecutive).  Runs after the SCF loop; neither timed nor counted as SCF launches.
static int export_radial(dftatom_ctx* c, const GridDev& g, const ScfBuffers& b, const std::vector<AtomDev>& atoms, const RadialDest& rd)
{
    const dftatom_radial& R = *rd.rad;
    const int n_atoms = b.n_atoms, n_orbs = b.n_orbs;
    const size_t N = (size_t)g.N;
    cudaStream_t st = c->stream;
    const bool fields = R.rho || R.v || R.v_hartree || R.atom_moments, orbitals = R.orbitals || R.moments;
    const size_t o_rho = 0, o_v = o_rho + (size_t)n_atoms * 2 * N, o_vh = o_v + (size_t)n_atoms * 2 * N, o_am = o_vh + (size_t)n_atoms * N;
    const size_t o_u = o_am + (size_t)n_atoms * 2, o_mom = o_u + (size_t)n_orbs * N, total = o_mom + (size_t)n_orbs * DFTATOM_N_MOMENTS;
    const int rows = std::max(n_atoms, n_orbs);
    int rc;
    if ((rc = c->radial.ensure(sizeof(double) * total)) || (rc = c->radial_part.ensure(sizeof(double) * (size_t)radial_part_doubles(g.N, rows)))
        || (rc = c->radial_ticket.ensure(sizeof(int) * (size_t)rows))) return rc;
    double* sb = c->radial.as<double>();
    DFT_CHECK(cudaMemsetAsync(c->radial_ticket.p, 0, sizeof(int) * (size_t)rows, st));
    if (fields) launch_radial_fields(g, b, sb + o_rho, sb + o_v, sb + o_vh, sb + o_am, c->radial_part.as<double>(), c->radial_ticket.as<int>(), st);
    if (orbitals) launch_radial_orbitals(g, b.psi, b.inv_norm, 1, n_orbs, sb + o_u, sb + o_mom, c->radial_part.as<double>(), c->radial_ticket.as<int>(), st);
    long long bytes = 0;
    auto copy = [&](double* dst, const double* src, size_t n) -> int {
        DFT_CHECK(cudaMemcpyAsync(dst, src, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
        bytes += (long long)(sizeof(double) * n);
        return 0;
    };
    if (rd.copy_r && R.r && (rc = copy(R.r, g.r, N))) return rc;
    for (int a0 = 0, a1; a0 < n_atoms; a0 = a1) {
        int n_rows = atoms[a0].orb_count[0] + atoms[a0].orb_count[1];
        for (a1 = a0 + 1; a1 < n_atoms && rd.atom[a1] == rd.atom[a1 - 1] + 1; ++a1) n_rows += atoms[a1].orb_count[0] + atoms[a1].orb_count[1];
        const size_t na = (size_t)(a1 - a0), d = (size_t)rd.atom[a0], o0 = (size_t)atoms[a0].orb_begin[0], r0 = (size_t)rd.row[a0];
        if (R.rho && (rc = copy(R.rho + d * 2 * N, sb + o_rho + a0 * 2 * N, na * 2 * N))) return rc;
        if (R.v && (rc = copy(R.v + d * 2 * N, sb + o_v + a0 * 2 * N, na * 2 * N))) return rc;
        if (R.v_hartree && (rc = copy(R.v_hartree + d * N, sb + o_vh + a0 * N, na * N))) return rc;
        if (R.atom_moments && (rc = copy(R.atom_moments + d * 2, sb + o_am + a0 * 2, na * 2))) return rc;
        if (R.orbitals && (rc = copy(R.orbitals + r0 * N, sb + o_u + o0 * N, (size_t)n_rows * N))) return rc;
        if (R.moments && (rc = copy(R.moments + r0 * DFTATOM_N_MOMENTS, sb + o_mom + o0 * DFTATOM_N_MOMENTS, (size_t)n_rows * DFTATOM_N_MOMENTS))) return rc;
    }
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    c->last_d2h_bytes += bytes;
    return 0;
}

// A group of pseudo-atoms (dftatom_solve_pseudo_batch, validated there): the HOST ionic potentials and the atoms' descriptors
struct PseudoGroup {
    const double* v_ion; int n_rows;
    const dftatom_pseudo_atom* atoms;
    const double* rho_pc; int n_pc_rows;      // partial cores (dftatom_solve_pseudo_batch_core); NULL when no atom has one
    const int* pc_row;                        // [n_atoms], -1 = none (only read with rho_pc)
};

// The three ways of a warm Poisson solve in increment form (selected by solve_group's poisson_solve; dftatom_poisson_increment's `solver`)
enum { kIncDirect = 0, kIncWarmVcycles = 1, kIncColdForm = 2 };

// One warm Poisson solve in increment form of the densities ca.rho: A dU = S(rho) - S(rho_prev) with dU = 0 at both ends, U += dU,
// rho_prev = rho (ca.rho_prev, ca.U, ca.skip; ca.ldU is the row stride of U, d_src and d_u).  path kIncDirect: poisson_direct.cu (d_u is its
// scratch above 14 levels); kIncWarmVcycles: n_vcycles V-cycles of poisson_warm.cu in pa's hierarchy; kIncColdForm: n_vcycles V-cycles of
// the cold solvers (sa and splan: the stream solver when `stream`; else pa: poisson_full_kernel) on (d_src, d_u) between
// poisson_delta_prepare and poisson_delta_apply.  Shared by the SCF and dftatom_poisson_increment.
static void poisson_increment(int path, const GridDev& g, const PoissonLevels& lv, bool stream, const StreamPlan& splan, WarmPoissonArgs ca,
                              const PoissonArgs& pa, const StreamSolveArgs& sa, double* d_src, double* d_u, int n_vcycles, cudaStream_t st,
                              long long& n_launch)
{
    const int n_dens = ca.n_dens;
    const long long ldU = ca.ldU;
    ca.work = pa.work;
    if (path == kIncDirect) {
        ca.scratch = d_u; ca.scratch_stride = ldU;
        launch_poisson_direct(g, ca, st);
        ++n_launch;
    } else if (path == kIncWarmVcycles) {
        ca.n_vcycles = n_vcycles;
        launch_poisson_warm(g, ca, pa.phi, pa.src, lv.total, st);
        ++n_launch;
    } else {
        // increment form around the existing solvers: dS, dU = 0 -> V-cycles on (dS, dU) with zero boundary values -> U += dU
        launch_poisson_delta_prepare(g, n_dens, ldU, ca.rho, ca.rho_prev, d_src, d_u, ca.skip, ca.skip_stride_bytes, st);
        if (stream) {
            StreamSolveArgs sd = sa;
            sd.rho = nullptr; sd.src0 = d_src; sd.U = d_u; sd.Zbc = nullptr; sd.warm = 1; sd.n_v = n_vcycles;
            long long nl = 0;
            launch_poisson_stream_solve(splan, g.delta, sd, st, &nl);
            n_launch += nl;
        } else {
            PoissonArgs pd = pa;
            pd.rho = nullptr; pd.src_nat = d_src; pd.u_out = d_u; pd.nat_stride = ldU == g.N ? 0 : ldU; pd.Zbc = nullptr; pd.warm_vcycles = n_vcycles;
            // (team mode keeps Phi_0 in place in the hierarchy between warm solves: it must start from the zero increment too)
            cudaMemsetAsync(pa.phi, 0, sizeof(double) * (size_t)n_dens * lv.total, st);
            launch_poisson_full(g, lv, pd, st);
            ++n_launch;
        }
        launch_poisson_delta_apply(g, n_dens, ldU, ca.U, d_u, ca.skip, ca.skip_stride_bytes, st);
        n_launch += 2;
    }
}

// one group of atoms: its whole SCF, enqueued on the context's stream (pg: pseudo-atoms, opts[a].Z = their Z_b).  The callers have
// validated every atom's options and checked that all atoms share atom 0's grid.
static int solve_group(dftatom_ctx* c, const dftatom_options* opts, const dftatom_config* cfgs, int n_atoms, dftatom_result* out,
                       dftatom_step* steps, int steps_stride, const RadialDest* rd = nullptr, const PseudoGroup* pg = nullptr)
{
    if (!c || !opts || !out || n_atoms <= 0) { set_error("bad argument"); return DFTATOM_E_ARG; }
    const bool host_dbg = getenv("DFTATOM_DEBUG_HOST") != nullptr;      // development aid: wall-clock of the host-side stages
    auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double th0 = now();
    double th1 = 0., th2 = 0., th3 = 0., th4 = 0.;
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp = nullptr;
    GridEntry* gentry = nullptr;
    int rc = get_grid(c, opts[0].levels, opts[0].method >= 2 ? 0. : opts[0].delta, opts[0].max_r, &gp, &gentry);
    if (rc) return rc;
    const GridDev g = *gp;
    const int N = g.N;
    const PoissonLevels lv = make_levels(g.L);
    cudaStream_t st = c->stream;

    // ---- host-side rules: levels per atom / spin ----
    std::vector<AtomDev> atoms(n_atoms);
    std::vector<AtomState> astate(n_atoms);
    std::vector<OrbitalDev> orbs;
    std::vector<int> tab_of(2 * (size_t)n_atoms, -1);
    std::vector<double> zbc(n_atoms);
    std::vector<std::vector<dftatom_level>> lev_a(n_atoms), lev_b(n_atoms);
    std::vector<PseudoAtomDev> patoms(pg ? n_atoms : 0);
    int n_tabs = 0, max_steps = 0, zmax = 1;
    for (int a = 0; a < n_atoms; ++a) {
        AtomDev& at = atoms[a];
        at.Z = opts[a].Z; at.method = opts[a].method & 1; at.n_spin = at.method ? 2 : 1;       // 0 / 2: LDA, 1 / 3: LSDA
        at.n_steps_max = at.method ? DFTATOM_MAX_STEPS_LSDA : DFTATOM_MAX_STEPS_LDA;            // DFTAtom.cpp:106 / :699 (same caps as :396 / :908)
        if (c->k.step_cap > 0) at.n_steps_max = std::min(at.n_steps_max, c->k.step_cap);
        at.mixing = opts[a].mixing;
        max_steps = std::max(max_steps, at.n_steps_max);
        zmax = std::max(zmax, at.Z);
        AtomLevels al;
        if ((rc = atom_levels(a, opts[a], cfgs ? &cfgs[a] : nullptr, &al, pg ? pg->atoms[a].z_val : 0.))) return rc;
        if (pg) for (auto& L : al.lev) for (dftatom_level& x : L) x.nodes = x.n - pg->atoms[a].n_ref[x.l];
        lev_a[a] = al.lev[0]; lev_b[a] = al.lev[1];
        at.n_el[0] = al.n_el[0]; at.n_el[1] = al.n_el[1];
        zbc[a] = al.n_el[0] + al.n_el[1];                    // U(Rmax) = the electron count Q (Z for the neutral atom)
        for (int s = 0; s < at.n_spin; ++s) {
            tab_of[2 * a + s] = n_tabs;
            at.orb_begin[s] = (int)orbs.size();
            const auto& L = al.lev[s];
            at.orb_count[s] = (int)L.size();
            for (size_t k = 0; k < L.size(); ++k) {
                OrbitalDev o; o.atom = a; o.spin = s; o.n0 = L[k].n - 1; o.l = L[k].l; o.occ = al.occ[s][k]; o.want = L[k].nodes; o.tab = n_tabs;
                orbs.push_back(o);
            }
            ++n_tabs;
        }
        if (at.n_spin == 1) { at.orb_begin[1] = 0; at.orb_count[1] = 0; }
        if (pg) {       // one row per (spin, channel) after the atom's density rows; its orbitals are solved in the row of their l
            PseudoAtomDev& p = patoms[a];
            for (int l = 0; l < 4; ++l) {
                p.vrow[l] = pg->atoms[a].row[l];
                for (int s = 0; s < 2; ++s) p.tab[s][l] = (p.vrow[l] >= 0 && s < at.n_spin) ? n_tabs++ : -1;
            }
            for (size_t q = (size_t)at.orb_begin[0]; q < orbs.size(); ++q) orbs[q].tab = p.tab[orbs[q].spin][orbs[q].l];
        }
        astate[a] = AtomState{ 0., 0, 0, 0, DFTATOM_MAX_STEPS, opts[a].mixing, 0., 0., 0, 0 };
    }
    const int n_orbs = (int)orbs.size();
    const int stride = max_steps;
    c->last_graph_iterations = 0;
    c->last_h2d_bytes = (long long)(sizeof(AtomDev) * atoms.size() + sizeof(AtomState) * astate.size() + sizeof(OrbitalDev) * orbs.size()
                                    + sizeof(int) * (tab_of.size() + 2) + sizeof(double) * zbc.size());

    const bool core = pg && pg->rho_pc;
    const size_t pseudo_bytes = pg ? sizeof(PseudoAtomDev) * patoms.size() + sizeof(double) * (size_t)pg->n_rows * N
                                     + (core ? sizeof(double) * (size_t)pg->n_pc_rows * N + sizeof(int) * (size_t)n_atoms : 0) : 0;

    // ---- device buffers ----
    if ((rc = upload_arena_reset(c, (size_t)c->last_h2d_bytes + pseudo_bytes + 64 * 8))) return rc;
    if ((rc = upload(c, c->atoms, atoms))) return rc;
    if ((rc = upload(c, c->astate, astate))) return rc;
    if ((rc = upload(c, c->orbs, orbs))) return rc;
    if ((rc = upload(c, c->tab_of, tab_of))) return rc;
    if ((rc = upload(c, c->zbc, zbc))) return rc;
    if ((rc = c->ss.ensure(sizeof(SearchState) * (size_t)n_orbs))) return rc;
    if ((rc = c->rho.ensure(sizeof(double) * (size_t)n_tabs * N))) return rc;
    if ((rc = c->rhot.ensure(sizeof(double) * (size_t)n_atoms * N))) return rc;
    if ((rc = c->vpot.ensure(sizeof(double) * (size_t)n_tabs * N))) return rc;
    if ((rc = c->atab.ensure(sizeof(double) * (size_t)n_tabs * N))) return rc;
    if ((rc = c->psi.ensure(sizeof(double) * (size_t)n_orbs * N))) return rc;
    if ((rc = c->match_pt.ensure(sizeof(int) * (size_t)n_orbs))) return rc;
    if ((rc = c->inv_norm.ensure(sizeof(double) * (size_t)n_orbs))) return rc;
    if ((rc = c->epart.ensure(sizeof(double) * (size_t)n_atoms * 64 * (core ? 6 : 5))) || (rc = c->eticket.ensure(sizeof(int) * (size_t)n_atoms))) return rc;
    DFT_CHECK(cudaMemsetAsync(c->eticket.p, 0, sizeof(int) * (size_t)n_atoms, st));
    if ((rc = c->phi.ensure(sizeof(double) * (size_t)n_atoms * lv.total))) return rc;
    if ((rc = c->src.ensure(sizeof(double) * (size_t)n_atoms * lv.total))) return rc;
    if ((rc = c->u0.ensure(sizeof(double) * (size_t)n_atoms * N))) return rc;
    if (n_atoms > 65535) { set_error("at most 65535 atoms per batch"); return DFTATOM_E_ARG; }      // gridDim.y of the per-density launches
    const bool exact = c->k.poisson_exact != 0;
    const bool stream = !exact && c->k.stream_poisson && n_atoms >= c->k.stream_min_dens && g.L >= c->k.stream_min_levels && g.L > c->k.stream_mid_levels && g.L <= 22 && c->k.refine_vcycles == 0 && !c->k.floor_stop;
    const int ldU = stream ? ((N + 3) & ~3) : N;
    const StreamPlan splan = stream ? make_stream_plan(g.L, n_atoms, c->k.stream_mid_levels) : StreamPlan{};
    if ((rc = c->ubuf.ensure(sizeof(double) * (size_t)n_atoms * ldU))) return rc;
    if (stream && ((rc = c->stream_src0.ensure(sizeof(double) * (size_t)n_atoms * ldU)) || (rc = c->stream_scratch.ensure(sizeof(double) * (size_t)splan.total)))) return rc;
    if (exact && (rc = c->exact_work.ensure(sizeof(double) * (size_t)n_atoms * (size_t)exact_poisson_work_doubles(g.L)))) return rc;
    const bool delta = c->k.delta_poisson && !exact && c->k.warm_vcycles > 0 && c->k.refine_vcycles == 0 && !c->k.floor_stop;
    if (delta && ((rc = c->rho_prev.ensure(sizeof(double) * (size_t)n_atoms * N)) || (rc = c->d_src.ensure(sizeof(double) * (size_t)n_atoms * ldU))
                  || (rc = c->d_u.ensure(sizeof(double) * (size_t)n_atoms * ldU)))) return rc;
    if ((rc = c->steps.ensure(sizeof(dftatom_step) * (size_t)n_atoms * stride))) return rc;
    if ((rc = c->last_steps.ensure(sizeof(dftatom_step) * (size_t)n_atoms))) return rc;
    if ((rc = c->n_active.ensure(sizeof(int) * 2))) return rc;
    PseudoArgs pargs{};
    if (pg) {
        if ((rc = upload(c, c->pseudo_atoms, patoms))) return rc;
        if ((rc = upload(c, c->pseudo_v, std::vector<double>(pg->v_ion, pg->v_ion + (size_t)pg->n_rows * N)))) return rc;
        pargs.atoms = c->pseudo_atoms.as<PseudoAtomDev>(); pargs.v_ion = c->pseudo_v.as<double>();
        if (core) {
            if ((rc = upload(c, c->pseudo_pc, std::vector<double>(pg->rho_pc, pg->rho_pc + (size_t)pg->n_pc_rows * N)))) return rc;
            if ((rc = upload(c, c->pseudo_pc_row, std::vector<int>(pg->pc_row, pg->pc_row + n_atoms)))) return rc;
            pargs.rho_pc = c->pseudo_pc.as<double>(); pargs.pc_row = c->pseudo_pc_row.as<int>();
        }
        c->last_h2d_bytes += (long long)pseudo_bytes;
    }
    DFT_CHECK(cudaMemsetAsync(c->steps.p, 0, sizeof(dftatom_step) * (size_t)n_atoms * stride, st));
    DFT_CHECK(cudaMemsetAsync(c->ss.p, 0, sizeof(SearchState) * (size_t)n_orbs, st));
    const int h_counts[2] = { n_atoms, n_orbs };        // atoms / orbitals still iterating, kept up to date by potential_energy_kernel
    DFT_CHECK(cudaMemcpyAsync(c->n_active.p, h_counts, sizeof(int) * 2, cudaMemcpyHostToDevice, st));

    ScfBuffers b{};
    b.n_atoms = n_atoms; b.n_orbs = n_orbs; b.n_tabs = n_tabs; b.N = N;
    b.atoms = c->atoms.as<AtomDev>(); b.astate = c->astate.as<AtomState>(); b.orbs = c->orbs.as<OrbitalDev>();
    b.ss = c->ss.as<SearchState>(); b.rho = c->rho.as<double>(); b.rhot = c->rhot.as<double>(); b.vpot = c->vpot.as<double>();
    b.atab = c->atab.as<double>(); b.psi = c->psi.as<double>(); b.match_pt = c->match_pt.as<int>(); b.inv_norm = c->inv_norm.as<double>(); b.epart = c->epart.as<double>(); b.eticket = c->eticket.as<int>();
    b.phi = c->phi.as<double>(); b.src = c->src.as<double>(); b.U = c->ubuf.as<double>(); b.ldU = ldU; b.Zbc = c->zbc.as<double>(); b.tab_of = c->tab_of.as<int>();
    b.steps = c->steps.as<dftatom_step>(); b.steps_stride = stride; b.n_active = c->n_active.as<int>();
    b.run_to_cap = c->k.run_to_cap; b.adaptive_mixing = c->k.adaptive_mixing;

    PoissonArgs pa{};
    pa.n_dens = n_atoms; pa.rho = b.rhot; pa.Zbc = b.Zbc; pa.phi = b.phi; pa.src = b.src; pa.u_out = b.U; pa.coarse_op = g.coarse_op;
    pa.skip = &b.astate[0].done; pa.skip_stride_bytes = (int)sizeof(AtomState);
    pa.max_vcycles = c->k.max_vcycles; pa.floor_stop = c->k.floor_stop;
    pa.refine_vcycles = c->k.refine_vcycles; pa.u0 = c->u0.as<double>();
    if ((rc = c->team_bar.ensure(sizeof(unsigned) * (size_t)n_atoms))) return rc;
    pa.team_bar = c->k.team_poisson ? c->team_bar.as<unsigned>() : nullptr;
    pa.nat_stride = 0; pa.n_sm = c->n_sm;
    ExactPoissonArgs xa{};
    xa.n_dens = n_atoms; xa.L = g.L; xa.delta = g.delta; xa.rho = b.rhot; xa.rho_stride = N; xa.r = g.r; xa.pex = g.pex; xa.Zbc = b.Zbc;
    xa.U = b.U; xa.ldU = ldU; xa.work = c->exact_work.as<double>(); xa.skip = &b.astate[0].done; xa.skip_stride_bytes = (int)sizeof(AtomState);
    xa.max_vcycles = 100;                                       // PoissonSolver.h:117
    WarmPoissonArgs ca{};
    ca.n_dens = n_atoms; ca.rho = b.rhot; ca.rho_stride = N; ca.U = b.U; ca.ldU = ldU; ca.Zbc = b.Zbc; ca.coarse_tri = g.coarse_tri;
    ca.skip = &b.astate[0].done; ca.skip_stride_bytes = (int)sizeof(AtomState); ca.rho_prev = c->rho_prev.as<double>();
    StreamSolveArgs sa{};
    sa.n_dens = n_atoms; sa.rho = b.rhot; sa.rho_stride = N; sa.psrc = g.psrc; sa.src0 = c->stream_src0.as<double>(); sa.U = b.U; sa.ld0 = ldU;
    sa.Zbc = b.Zbc; sa.scratch = c->stream_scratch.as<double>(); sa.coarse_op = g.coarse_op; sa.variant = c->k.stream_variant;
    sa.skip = &b.astate[0].done; sa.skip_stride_bytes = (int)sizeof(AtomState);
    // the Poisson solve of one SCF step: FullCycle (ramp + max_vcycles V-cycles), or warm_vcycles V-cycles from the previous U
    double* rho_prev = c->rho_prev.as<double>();
    double* d_src = c->d_src.as<double>();
    double* d_u = c->d_u.as<double>();
    const int* skip_p = &b.astate[0].done; const int skip_stride = (int)sizeof(AtomState);
    const bool warm_ok = delta && !stream && poisson_warm_supported(g.L, g.delta) && g.coarse_tri != nullptr && (long long)lv.total >= poisson_warm_scratch_doubles(g.L);
    const bool direct_ok = c->k.direct_poisson && delta && g.coarse_direct != nullptr;
    int cur_step = 0;               // SCF step being enqueued (the graph body is captured at the first steady-state step)
    auto poisson_solve = [&](int warm_vcycles, long long& n_launch) {
        const bool warm = warm_vcycles > 0;
        if (exact) {
            launch_poisson_exact(xa, st);
            ++n_launch;
        } else if (warm && delta) {
            const int path = direct_ok && cur_step >= c->k.direct_after ? kIncDirect : warm_ok ? kIncWarmVcycles : kIncColdForm;
            poisson_increment(path, g, lv, stream, splan, ca, pa, sa, d_src, d_u, warm_vcycles, st, n_launch);
        } else if (stream) {
            sa.warm = warm; sa.n_v = warm ? warm_vcycles : c->k.max_vcycles;
            long long nl = 0;
            launch_poisson_stream_solve(splan, g.delta, sa, st, &nl);
            n_launch += nl;
        } else {
            pa.warm_vcycles = warm_vcycles;
            launch_poisson_full(g, lv, pa, st);
            ++n_launch;
        }
        if (delta && !warm) {       // a cold solve: remember its density for the first increment
            launch_poisson_delta_prepare(g, n_atoms, ldU, b.rhot, rho_prev, nullptr, nullptr, skip_p, skip_stride, st);
            ++n_launch;
        }
    };

    if (max_steps > 256) { set_error("internal: step cap"); return DFTATOM_E_ARG; }
    EventPool events;                       // destroyed on every return path
    cudaEvent_t ev0 = events.make(true), ev1 = events.make(true);
    std::vector<cudaEvent_t> step_ev(max_steps);
    for (auto& e : step_ev) e = events.make(false);
    if (!events.ok) { set_error("cudaEventCreate failed"); return DFTATOM_E_CUDA; }

    long long launches = 0;
    // optional per-class kernel timing: one event pair per launch group, resolved after the final sync
    struct Span { int cls; cudaEvent_t a, b; };
    std::vector<Span> spans;
    const bool prof = c->k.profile != 0;
    unsigned long long* d_work = nullptr;
    if ((rc = c->scratch[7].ensure(sizeof(unsigned long long) * 32))) return rc;
    d_work = c->scratch[7].as<unsigned long long>();
    DFT_CHECK(cudaMemsetAsync(d_work, 0, sizeof(unsigned long long) * 32, st));
    pa.work = d_work + DFTATOM_K_POISSON;
    // the event pairs of the per-class timing are created BEFORE the timed loop (profile = 1 must not put cudaEventCreate into it)
    std::vector<cudaEvent_t> span_ev;
    if (prof) { span_ev.resize((size_t)max_steps * DFTATOM_K_COUNT * 2); for (auto& e : span_ev) e = events.make(true); if (!events.ok) { set_error("cudaEventCreate failed"); return DFTATOM_E_CUDA; } }
    size_t span_next = 0;
    auto begin_span = [&](int cls) { if (prof) { Span s{ cls, span_ev[span_next], span_ev[span_next + 1] }; span_next += 2; cudaEventRecord(s.a, st); spans.push_back(s); } };
    auto end_span = [&]() { if (prof) cudaEventRecord(spans.back().b, st); };
    // NVTX ranges per SCF phase (host side: they bracket the enqueue of the phase's launches; SURVEY section 5)
    static const char* const kPhase[DFTATOM_K_COUNT] = { "dftatom:search", "dftatom:match", "dftatom:density", "dftatom:poisson", "dftatom:potential" };
    auto begin_phase = [&](int cls) { nvtxRangePushA(kPhase[cls]); begin_span(cls); };
    auto end_phase = [&]() { end_span(); nvtxRangePop(); };
    th1 = now();
    g_dft_pdl = c->k.use_pdl;
    DFT_CHECK(cudaEventRecord(ev0, st));
    // initial guess -> U -> V   (DFTAtom.cpp:371-392)
    launch_initial_density(g, b, st); ++launches;
    // The start density is n_el / volume on every node but the first and the boundary value is the electron count Q: A U = S is linear in
    // Q.  One cold solve of the Q = 1 problem per grid (the same kernel, the same cycle), U_atom = Q U_1 afterwards.
    const bool unit_guess = c->k.unit_guess && !exact && !stream && !g.uniform && g.L <= 14 && gentry != nullptr;
    if (unit_guess) {
        if (!gentry->u_unit_ok) {
            if ((rc = gentry->u_unit.ensure(sizeof(double) * (size_t)(2 * N + 2)))) return rc;
            double* u1 = gentry->u_unit.as<double>();
            double* rho1 = u1 + N;
            double* one = rho1 + N;
            std::vector<double> h1((size_t)N, 1. / (4. * M_PI / 3. * g.max_r * g.max_r * g.max_r));
            h1[0] = 0.;
            const double h_one = 1.;
            DFT_CHECK(cudaMemcpyAsync(rho1, h1.data(), sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, st));
            DFT_CHECK(cudaMemcpyAsync(one, &h_one, sizeof(double), cudaMemcpyHostToDevice, st));
            DFT_CHECK(cudaStreamSynchronize(st));                       // (h1, h_one are pageable locals)
            PoissonArgs p1 = pa;
            p1.n_dens = 1; p1.rho = rho1; p1.src_nat = nullptr; p1.u_out = u1; p1.nat_stride = 0; p1.Zbc = one; p1.skip = nullptr; p1.skip_stride_bytes = 0;
            p1.warm_vcycles = 0; p1.team_bar = nullptr;
            launch_poisson_full(g, lv, p1, st); ++launches;
            gentry->u_unit_ok = true;
        }
        launch_scale_unit_potential(g.N, n_atoms, ldU, gentry->u_unit.as<double>(), b.Zbc, b.U, st); ++launches;
        if (delta) { launch_poisson_delta_prepare(g, n_atoms, ldU, b.rhot, rho_prev, nullptr, nullptr, skip_p, skip_stride, st); ++launches; }
    } else {
        poisson_solve(0, launches);
    }
    if (pg) launch_pseudo_potential_energy(g, b, pargs, 1, st);
    else launch_potential_energy(g, lv, b, 1, st);
    ++launches;

    const int rounds = search_rounds_needed(zmax);
    int steps_enqueued = 0;
    const int lag = 2;
    // one SCF step = five kernel classes enqueued on the stream; nothing in it touches the host
    // sp: the SCF step being enqueued; [sp, sp_end): the steps these launches may be executed at (a graph body is replayed for a range of steps)
    auto enqueue_step = [&](int sp, int sp_end, long long& nl) {
        nvtxRangePushA("dftatom:scf_step");
        begin_phase(DFTATOM_K_SEARCH);
        if (c->k.search_mode == 0 && c->k.search_kernel == 0 && !g.uniform) {
            nl += launch_search_rows(g, b.atab, b.atoms, b.orbs, b.astate, b.ss, n_orbs, d_work + DFTATOM_K_SEARCH, (c->k.warm_start ? 1 : 0) | (c->k.search_predict ? 2 : 0), c->k.rows_cfg, c->k.rows_wide_from_step, sp, sp_end, st);
        } else if (c->k.search_mode == 0) {
            // two shapes of the same search: serial-in-r (one warp per orbital) while many orbitals are active, parallel-in-r
            // (one cluster per orbital) once few are left.  Both are enqueued; the device-side count of active orbitals
            // decides which one runs (the other returns at once), so the host never has to know.
            const int segs = c->segments(N);
            const int thr = segs > 1 ? c->k.seg_threshold : -1;
            const bool serial_too = !(segs > 1 && c->k.seg_threshold >= n_orbs);      // the serial-in-r kernel can never be selected: do not launch it
            if (serial_too) {
                launch_search_fused(g, b.atab, b.atoms, b.orbs, b.astate, b.ss, n_orbs, d_work + DFTATOM_K_SEARCH, b.n_active + 1, thr, c->k.warm_start, st);
                ++nl;
            }
            if (segs > 1) {
                launch_search_seg(g, b.atab, b.atoms, b.orbs, b.astate, b.ss, n_orbs, d_work + DFTATOM_K_SEARCH, segs, b.n_active + 1, thr, c->k.warm_start, st);
                ++nl;
            }
        } else {
            launch_search_init(g, b.atoms, b.astate, b.orbs, b.ss, n_orbs, st); ++nl;
        }
        if (c->k.search_mode != 0) for (int r = 0; r < rounds; ++r) { launch_search_round(g, b.atab, b.orbs, b.astate, b.ss, n_orbs, d_work + DFTATOM_K_SEARCH, st); ++nl; }
        end_phase();
        begin_phase(DFTATOM_K_MATCH);
        if (c->k.match_mode == 0) nl += launch_match_cta(g, b.atab, b.orbs, b.astate, b.ss, b.psi, b.match_pt, b.inv_norm, n_orbs, c->k.match_win_until_step, c->k.match_win_nodes, sp, sp_end, st);
        else {                                              // validation paths: warp-per-orbital / reference-shaped serial solution
            if (c->k.match_mode == 2) launch_match_seg(g, b.atab, b.orbs, b.astate, b.ss, b.psi, b.match_pt, n_orbs, st);
            else launch_match(g, b.atab, b.orbs, b.astate, b.ss, b.psi, b.match_pt, n_orbs, st);
            launch_orbital_norms(g, b, st); nl += 2;
        }
        end_phase();
        begin_phase(DFTATOM_K_DENSITY);
        launch_density_update(g, b, st); ++nl;
        end_phase();
        begin_phase(DFTATOM_K_POISSON);
        cur_step = sp;
        poisson_solve(sp >= c->k.warm_after ? c->k.warm_vcycles : 0, nl);
        end_phase();
        begin_phase(DFTATOM_K_POTENTIAL);
        if (pg) launch_pseudo_potential_energy(g, b, pargs, 0, st);
        else launch_potential_energy(g, lv, b, 0, st);
        ++nl;
        end_phase();
        nvtxRangePop();
    };
    // The SCF loop.  Default: the steady-state step (from step warm_after on every step enqueues the same launches) is captured ONCE into
    // the body of a CUDA-graph WHILE node whose condition - "some atom is still iterating" - is set on the device by the last kernel of the
    // body (cudaGraphSetConditional): one graph launch runs the rest of the SCF of the whole batch with no host round trip at all.
    // Not used with per-class event timing (profile), the validation search / match modes, or the cooperative team-mode Poisson kernel.
    const bool team_possible = g.L >= 15 && !stream && !exact;
    const bool graph_ok = c->k.use_graph && !prof && c->k.search_mode == 0 && c->k.match_mode == 0 && (!team_possible || direct_ok);
    bool graph_done = false;
    if (graph_ok) {
        const int n_cold = std::min(max_steps, std::max(std::max(0, c->k.warm_after), direct_ok ? c->k.direct_after : 0));
        for (int sp = 0; sp < n_cold; ++sp) { enqueue_step(sp, sp + 1, launches); ++steps_enqueued; }
        if (n_cold < max_steps) {
            // phases: the ranges of SCF steps between the step indices at which a kernel shape hands over to another one
            std::vector<int> cut{ n_cold };
            if (c->k.graph_phases && c->k.search_kernel == 0 && !g.uniform) {
                for (int s_ : { c->k.rows_wide_from_step, c->k.match_win_until_step })
                    if (s_ > n_cold && s_ < max_steps && std::find(cut.begin(), cut.end(), s_) == cut.end()) cut.push_back(s_);
                std::sort(cut.begin(), cut.end());
            }
            cut.push_back(1 << 30);
            ScfLoopPhases ph{};
            ph.n = (int)cut.size() - 1;                 // <= 3
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            long long per_iter[4] = {};
            bool ok = cudaGraphCreate(&graph, 0) == cudaSuccess;
            // every handle first: the condition kernel of a phase also switches the later phases off
            for (int p_ = 0; ok && p_ < ph.n; ++p_) ok = cudaGraphConditionalHandleCreate(&ph.handle[p_], graph, 1, cudaGraphCondAssignDefault) == cudaSuccess;
            cudaGraphNode_t prev_node = nullptr;
            for (int p_ = 0; ok && p_ < ph.n; ++p_) {
                cudaGraphNodeParams np = {};
                np.type = cudaGraphNodeTypeConditional;
                np.conditional.handle = ph.handle[p_]; np.conditional.type = cudaGraphCondTypeWhile; np.conditional.size = 1;
                cudaGraphNode_t node;
                ok = cudaGraphAddNode(&node, graph, prev_node ? &prev_node : nullptr, prev_node ? 1 : 0, &np) == cudaSuccess;
                if (!ok) break;
                prev_node = node;
                cudaGraph_t body = np.conditional.phGraph_out[0];
                ok = cudaStreamBeginCaptureToGraph(st, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
                if (ok) {
                    enqueue_step(cut[p_], cut[p_ + 1], per_iter[p_]);
                    launch_scf_loop_condition(ph, p_, n_cold, cut[p_ + 1], b.n_active, d_work + 6, st); ++per_iter[p_];
                    ok = cudaStreamEndCapture(st, nullptr) == cudaSuccess;
                }
            }
            ok = ok && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
            th2 = now();
            if (ok) {
                ok = cudaGraphLaunch(exec, st) == cudaSuccess;
                graph_done = ok;
            }
            if (graph_done) {
                DFT_CHECK(cudaStreamSynchronize(st));
                unsigned long long iters = 0;
                DFT_CHECK(cudaMemcpy(&iters, d_work + 6, sizeof(iters), cudaMemcpyDeviceToHost));
                for (int p_ = 0; p_ < ph.n; ++p_) {        // iterations of phase p: the steps of [cut[p], cut[p + 1]) that were executed
                    const long long first = cut[p_] - n_cold, last = std::min<long long>((long long)iters, (long long)cut[p_ + 1] - n_cold);
                    if (last > first) launches += per_iter[p_] * (last - first);
                }
                steps_enqueued += (int)iters;
                c->last_graph_iterations = (long long)iters;
            }
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
            if (!graph_done) { cudaGetLastError(); set_error("CUDA graph construction failed"); return DFTATOM_E_CUDA; }
        } else graph_done = true;
    }
    for (int sp = graph_done ? max_steps : 0; sp < max_steps; ++sp) {
        enqueue_step(sp, sp + 1, launches);
        DFT_CHECK(cudaMemcpyAsync(&c->h_active[sp], b.n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
        DFT_CHECK(cudaEventRecord(step_ev[sp], st));
        ++steps_enqueued;
        if (sp >= lag) {
            // the host stays `lag` steps ahead of the device: it never idles the GPU, it only stops enqueueing
            DFT_CHECK(cudaEventSynchronize(step_ev[sp - lag]));
            if (c->h_active[sp - lag] == 0) break;
        }
    }
    DFT_CHECK(cudaEventRecord(ev1, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    th3 = now();
    float ms = 0.f;
    DFT_CHECK(cudaEventElapsedTime(&ms, ev0, ev1));
    c->last_ms = ms; c->last_launches = launches;
    {
        unsigned long long hw[32] = {};
        DFT_CHECK(cudaMemcpy(hw, d_work, sizeof(hw), cudaMemcpyDeviceToHost));
        if (prof && getenv("DFTATOM_DEBUG_ROUNDS")) {
            fprintf(stderr, "search rounds histogram (orbital solves with r rounds, r = 1..15+):");
            for (int r = 1; r < 16; ++r) fprintf(stderr, " %llu", hw[8 + r]);
            fprintf(stderr, "\n  rounds summed per l = s p d f: %llu %llu %llu %llu;  solves with >= 4 rounds per l: %llu %llu %llu %llu\n", hw[24], hw[25], hw[26], hw[27],
                    hw[28], hw[29], hw[30], hw[31]);
        }
        for (int k = 0; k < DFTATOM_K_COUNT; ++k) { c->prof[k].ms = 0.; c->prof[k].launches = 0; c->prof[k].work = (double)hw[k]; }
        const bool step_dbg = prof && getenv("DFTATOM_DEBUG_STEPS");          // development aid: per-step time of every kernel class
        size_t span_i = 0;
        for (Span& s : spans) {
            float t = 0.f;
            cudaEventElapsedTime(&t, s.a, s.b);
            if (step_dbg) {
                const size_t sp = span_i / DFTATOM_K_COUNT;
                if (span_i % DFTATOM_K_COUNT == 0) fprintf(stderr, "step %3zu active %4d |", sp, sp < 256 ? c->h_active[sp] : -1);
                fprintf(stderr, " %s %.1f us", kPhase[s.cls] + 8, 1e3 * t);
                if (span_i % DFTATOM_K_COUNT == DFTATOM_K_COUNT - 1) fprintf(stderr, "\n");
            }
            ++span_i;
            c->prof[s.cls].ms += t;
            const bool rows = c->k.search_mode == 0 && c->k.search_kernel == 0 && !g.uniform;
            c->prof[s.cls].launches += (s.cls == DFTATOM_K_SEARCH) ? (rows ? 1 : c->k.search_mode == 0 ? ((c->segments(N) > 1 && c->k.seg_threshold < n_orbs) ? 2 : 1) : rounds + 1) : 1;
        }
    }

    // ---- results ----
    // Download what the caller asked for: with steps == NULL only the last record of every atom (gathered on the device,
    // n_atoms records) instead of the whole [n_atoms][stride] step array.
    const size_t n_rec = steps ? (size_t)n_atoms * stride : (size_t)n_atoms;
    if (n_rec > c->h_last_cap) {
        if (c->h_last) cudaFreeHost(c->h_last);
        c->h_last = nullptr; c->h_last_cap = 0;
        DFT_CHECK(cudaMallocHost((void**)&c->h_last, sizeof(dftatom_step) * n_rec));
        c->h_last_cap = n_rec;
    }
    if (!steps) launch_gather_last_steps(b, c->last_steps.as<dftatom_step>(), st);
    DFT_CHECK(cudaMemcpyAsync(astate.data(), b.astate, sizeof(AtomState) * n_atoms, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(c->h_last, steps ? (const void*)b.steps : c->last_steps.p, sizeof(dftatom_step) * n_rec, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    c->last_d2h_bytes = (long long)(sizeof(AtomState) * n_atoms + sizeof(dftatom_step) * n_rec);
    for (int a = 0; a < n_atoms; ++a) {
        dftatom_result& R = out[a];
        std::memset(&R, 0, sizeof(R));
        R.status = astate[a].status;
        R.n_steps = astate[a].n_steps;
        R.n_spin = atoms[a].n_spin;
        const dftatom_step& last = steps ? c->h_last[(size_t)a * stride + std::max(0, R.n_steps - 1)] : c->h_last[a];
        for (int s = 0; s < R.n_spin; ++s) {
            const auto& L = s ? lev_b[a] : lev_a[a];
            R.n_levels[s] = (int)L.size();
            for (size_t k = 0; k < L.size(); ++k) { R.levels[s][k] = L[k]; R.levels[s][k].E = last.E[s][k]; R.sorted[s][k] = R.levels[s][k]; }
            // std::sort by E (DFTAtom.cpp:487 / :1012-1013)
            std::sort(R.sorted[s], R.sorted[s] + L.size(), [](const dftatom_level& x, const dftatom_level& y) { return x.E < y.E; });
        }
        R.Etotal = last.Etotal; R.Ekin = last.Ekin; R.Ecoul = last.Ecoul; R.Eenuc = last.Eenuc; R.Exc = last.Exc;
        if (steps) {
            const int ncopy = std::min(steps_stride, stride);
            std::memcpy(steps + (size_t)a * steps_stride, &c->h_last[(size_t)a * stride], sizeof(dftatom_step) * ncopy);
        }
    }
    (void)steps_enqueued;
    if (rd && (rc = export_radial(c, g, b, atoms, *rd))) return rc;
    th4 = now();
    if (host_dbg) fprintf(stderr, "solve_group host stages: setup+uploads %.3f ms | cold steps + graph build %.3f ms | device loop %.3f ms | results %.3f ms | device time %.3f ms\n",
                          th1 - th0, (th2 > 0. ? th2 : th1) - th1, th3 - (th2 > 0. ? th2 : th1), th4 - th3, c->last_ms);
    return 0;
}

// Every kernel of the SCF chain of one atom depends on the previous one, and from the middle of a batch on most launches
// are latency-bound and leave SMs idle (the Poisson solve runs one CTA per density).  Atoms are independent, so a large
// batch is dealt into two groups whose chains are enqueued by two host threads on two streams: the search of one group
// overlaps the Poisson solve of the other.  Results are identical to the single-group run (no atom sees another).
int dftatom_solve_batch(dftatom_ctx* c, const dftatom_options* opts, int n_atoms, dftatom_result* out, dftatom_step* steps,
                        int steps_stride)
{
    return dftatom_solve_batch_radial(c, opts, n_atoms, out, steps, steps_stride, nullptr);
}

int dftatom_solve_batch_radial(dftatom_ctx* c, const dftatom_options* opts, int n_atoms, dftatom_result* out, dftatom_step* steps,
                               int steps_stride, const dftatom_radial* radial)
{
    return dftatom_solve_batch_config(c, opts, nullptr, n_atoms, out, steps, steps_stride, radial);
}

int dftatom_solve_batch_config(dftatom_ctx* c, const dftatom_options* opts, const dftatom_config* configs, int n_atoms, dftatom_result* out,
                               dftatom_step* steps, int steps_stride, const dftatom_radial* radial)
{
    if (!c || !opts || !out || n_atoms <= 0) { set_error("bad argument"); return DFTATOM_E_ARG; }
    // one pass over the batch before anything is solved: per atom its options, atom 0's grid, its levels (configuration) and orbital rows
    std::vector<long long> orb_rows;
    for (int a = 0; a < n_atoms; ++a) {
        int rc = validate(opts[a]);
        if (rc) return rc;
        // methods 2 / 3 (CalculateUniformLDA / LSDA, DFTAtom.h:15,18) run on the uniform grid: delta is not used (grid key: delta = 0)
        const bool uni_a = opts[a].method >= 2, uni_0 = opts[0].method >= 2;
        if (opts[a].levels != opts[0].levels || uni_a != uni_0 || (!uni_a && opts[a].delta != opts[0].delta) || opts[a].max_r != opts[0].max_r) {
            set_error("all atoms of one batch must share (levels, delta, max_r) and the kind of grid");
            return DFTATOM_E_MIXED_GRID;
        }
        AtomLevels al;
        if ((rc = atom_levels(a, opts[a], configs ? &configs[a] : nullptr, &al))) return rc;
        if (radial) orb_rows.push_back((long long)(al.lev[0].size() + al.lev[1].size()));
    }
    // radial export: the first orbital row of every atom in the caller's arrays
    std::vector<int> dest_atom;
    std::vector<long long> dest_row;
    if (radial) { int rc = batch_rows(*radial, orb_rows, dest_atom, dest_row); if (rc) return rc; }
    const RadialDest rd_all{ radial, dest_atom.data(), dest_row.data(), true };
    const RadialDest* rd = radial ? &rd_all : nullptr;
    if (c->stream_groups < 2 || n_atoms < 32) return solve_group(c, opts, configs, n_atoms, out, steps, steps_stride, rd);
    if (opts[0].levels > 14) return solve_group(c, opts, configs, n_atoms, out, steps, steps_stride, rd);      // (large grids: one group - the stream-mode Poisson solver wants all densities in one launch)
    // G groups: this context and a chain of G - 1 child contexts (each its own stream and buffers)
    const int G = std::min(c->stream_groups, std::max(1, n_atoms / 16));
    std::vector<dftatom_ctx*> ctxs(1, c);
    for (dftatom_ctx* p = c; (int)ctxs.size() < G; p = p->child) {
        if (!p->child) { int rc = dftatom_create(&p->child, c->device); if (rc) return rc; }
        p->child->k = c->k; p->child->stream_groups = 1;
        ctxs.push_back(p->child);
    }
    // deal the atoms in order of decreasing cost (orbital count ~ Z; LSDA doubles it) round-robin into the groups; a configured atom keeps the
    // key of its Z (it only balances the groups), so every batch of neutral atoms keeps its grouping
    std::vector<int> order(n_atoms);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return opts[x].Z * (1 + (opts[x].method & 1)) > opts[y].Z * (1 + (opts[y].method & 1)); });
    std::vector<std::vector<int>> idx(G);
    for (int q = 0; q < n_atoms; ++q) idx[q % G].push_back(order[q]);
    for (auto& v : idx) std::sort(v.begin(), v.end());
    std::vector<std::vector<dftatom_options>> gopts(G);
    std::vector<std::vector<dftatom_config>> gcfg(G);
    std::vector<std::vector<dftatom_result>> gout(G);
    std::vector<std::vector<dftatom_step>> gsteps(G);
    for (int gI = 0; gI < G; ++gI) {
        for (int a : idx[gI]) gopts[gI].push_back(opts[a]);
        if (configs) for (int a : idx[gI]) gcfg[gI].push_back(configs[a]);
        gout[gI].resize(idx[gI].size());
        if (steps) gsteps[gI].resize(idx[gI].size() * (size_t)steps_stride);
    }
    // radial export: every group scatters its atoms' arrays straight into the caller's, at their indices in the batch
    std::vector<std::vector<int>> gatom(G);
    std::vector<std::vector<long long>> grow(G);
    std::vector<RadialDest> grd(G);
    for (int gI = 0; gI < G && radial; ++gI) {
        for (int a : idx[gI]) { gatom[gI].push_back(a); grow[gI].push_back(dest_row[a]); }
        grd[gI] = RadialDest{ radial, gatom[gI].data(), grow[gI].data(), gI == 0 };
    }
    std::vector<int> rcs(G, 0);
    std::vector<std::string> errs(G);
    std::vector<std::thread> th;
    for (int gI = 1; gI < G; ++gI)
        th.emplace_back([&, gI]() {
            rcs[gI] = solve_group(ctxs[gI], gopts[gI].data(), configs ? gcfg[gI].data() : nullptr, (int)gopts[gI].size(), gout[gI].data(), steps ? gsteps[gI].data() : nullptr, steps_stride,
                                  radial ? &grd[gI] : nullptr);
            if (rcs[gI]) errs[gI] = g_err;
        });
    rcs[0] = solve_group(c, gopts[0].data(), configs ? gcfg[0].data() : nullptr, (int)gopts[0].size(), gout[0].data(), steps ? gsteps[0].data() : nullptr, steps_stride, radial ? &grd[0] : nullptr);
    for (auto& t : th) t.join();
    if (rcs[0]) return rcs[0];
    for (int gI = 1; gI < G; ++gI) if (rcs[gI]) { set_error(errs[gI]); return rcs[gI]; }
    for (int gI = 0; gI < G; ++gI)
        for (size_t q = 0; q < idx[gI].size(); ++q) {
            out[idx[gI][q]] = gout[gI][q];
            if (steps) std::memcpy(steps + (size_t)idx[gI][q] * steps_stride, &gsteps[gI][q * (size_t)steps_stride], sizeof(dftatom_step) * (size_t)steps_stride);
        }
    for (int gI = 1; gI < G; ++gI) {
        dftatom_ctx* ch = ctxs[gI];
        c->last_ms = std::max(c->last_ms, ch->last_ms);
        c->last_launches += ch->last_launches;
        c->last_graph_iterations += ch->last_graph_iterations;
        c->last_h2d_bytes += ch->last_h2d_bytes; c->last_d2h_bytes += ch->last_d2h_bytes;
        for (int k = 0; k < DFTATOM_K_COUNT; ++k) { c->prof[k].ms += ch->prof[k].ms; c->prof[k].launches += ch->prof[k].launches; c->prof[k].work += ch->prof[k].work; }
    }
    return 0;
}

int dftatom_solve_pseudo_batch(dftatom_ctx* c, int levels, double delta, double max_r, const double* v_ion, int n_rows,
                               const dftatom_pseudo_atom* atoms, const dftatom_config* configs, int n_atoms, dftatom_result* out,
                               dftatom_step* steps, int steps_stride, const dftatom_radial* radial)
{
    return dftatom_solve_pseudo_batch_core(c, levels, delta, max_r, v_ion, n_rows, atoms, configs, n_atoms, out, steps, steps_stride, radial,
                                           nullptr, 0, nullptr);
}

int dftatom_solve_pseudo_batch_core(dftatom_ctx* c, int levels, double delta, double max_r, const double* v_ion, int n_rows,
                                    const dftatom_pseudo_atom* atoms, const dftatom_config* configs, int n_atoms, dftatom_result* out,
                                    dftatom_step* steps, int steps_stride, const dftatom_radial* radial, const double* rho_pc,
                                    int n_pc_rows, const int* pc_row)
{
    if (!c || !v_ion || !atoms || !configs || !out) { set_error("dftatom_solve_pseudo_batch: NULL argument"); return DFTATOM_E_ARG; }
    if (n_rows < 1 || n_atoms < 1) { set_error("dftatom_solve_pseudo_batch: n_rows and n_atoms must be >= 1"); return DFTATOM_E_ARG; }
    if (delta == 0.) { set_error("dftatom_solve_pseudo_batch: the uniform grid (delta = 0) is not supported"); return DFTATOM_E_BAD_OPTION; }
    static const char* const fn = "dftatom_solve_pseudo_batch";
    const int N = (1 << std::min(std::max(levels, 0), 20)) + 1;
    std::vector<dftatom_options> opts(n_atoms);
    std::vector<char> row_ok(n_rows, 0);
    std::vector<long long> orb_rows;
    int rc;
    for (int a = 0; a < n_atoms; ++a) {
        const dftatom_pseudo_atom& pa = atoms[a];
        const std::string at_a = where(fn, "atom", a);
        if (pa.method != 0 && pa.method != 1) { set_error(at_a + "method must be 0 (LDA) or 1 (LSDA)"); return DFTATOM_E_BAD_OPTION; }
        dftatom_options& o = opts[a];
        o.Z = 1; o.levels = levels; o.max_r = max_r; o.delta = delta; o.mixing = pa.mixing; o.method = pa.method;
        if ((rc = validate(o))) { set_error(at_a + dftatom_last_error()); return rc; }
        if (!(std::isfinite(pa.z_val) && pa.z_val > 0.)) { set_error(at_a + "z_val must be finite and > 0"); return DFTATOM_E_BAD_OPTION; }
        int n_ch = 0;
        for (int l = 0; l < 4; ++l) {
            if (pa.row[l] < -1 || pa.row[l] >= n_rows) {
                set_error(at_a + "row[" + std::to_string(l) + "] = " + std::to_string(pa.row[l]) + " outside -1.." + std::to_string(n_rows - 1));
                return DFTATOM_E_BAD_OPTION;
            }
            if (pa.row[l] < 0) continue;
            ++n_ch;
            if (pa.n_ref[l] < l + 1 || pa.n_ref[l] > 8) {
                set_error(at_a + "n_ref[" + std::to_string(l) + "] = " + std::to_string(pa.n_ref[l]) + " outside " + std::to_string(l + 1) + "..8");
                return DFTATOM_E_BAD_OPTION;
            }
        }
        if (!n_ch) { set_error(at_a + "no channel (every row is -1)"); return DFTATOM_E_BAD_OPTION; }
        const dftatom_config& cf = configs[a];
        if (cf.n_orbitals == 0) { set_error(at_a + "empty configuration"); return DFTATOM_E_BAD_OPTION; }
        AtomLevels al;
        if ((rc = atom_levels(a, o, &cf, &al, pa.z_val))) { set_error(at_a + dftatom_last_error()); return rc; }
        for (int k = 0; k < cf.n_orbitals; ++k) {
            const dftatom_occupation& x = cf.orb[k];
            const std::string at = at_a + "configuration entry " + std::to_string(k) + " (n = " + std::to_string(x.n) + ", l = " + std::to_string(x.l) + "): ";
            if (pa.row[x.l] < 0) { set_error(at + "l has no channel"); return DFTATOM_E_BAD_OPTION; }
            if (x.n < pa.n_ref[x.l]) { set_error(at + "n below n_ref = " + std::to_string(pa.n_ref[x.l])); return DFTATOM_E_BAD_OPTION; }
        }
        orb_rows.push_back(cf.n_orbitals);
        // the bracket of the energy search: -Z_b^2 - 1 at least 10 Ha below the deepest ionic potential of the atom
        double vmin = INFINITY;
        for (int l = 0; l < 4; ++l) {
            if (pa.row[l] < 0) continue;
            const double* v = v_ion + (size_t)pa.row[l] * N;
            if (!row_ok[pa.row[l]]) {
                if (const int i = bad_node(v, N)) {
                    set_error(at_a + "v_ion row " + std::to_string(pa.row[l]) + " is not finite at node " + std::to_string(i));
                    return DFTATOM_E_BAD_OPTION;
                }
                row_ok[pa.row[l]] = 1;
            }
            for (int i = 1; i < N; ++i) vmin = std::min(vmin, v[i]);
        }
        o.Z = bracket_z(vmin, 10.);
        if (!o.Z) { set_error(at_a + "ionic potential too deep (min V_ion = " + std::to_string(vmin) + " below -118^2 + 9)"); return DFTATOM_E_BAD_OPTION; }
        if (pc_row && (pc_row[a] < -1 || pc_row[a] >= (rho_pc ? n_pc_rows : 0))) {
            set_error(at_a + "pc_row = " + std::to_string(pc_row[a]) + " outside -1.." + std::to_string((rho_pc ? n_pc_rows : 0) - 1));
            return DFTATOM_E_BAD_OPTION;
        }
    }
    bool any_core = false;
    for (int a = 0; pc_row && a < n_atoms; ++a) any_core |= pc_row[a] >= 0;
    for (int q = 0; any_core && q < n_pc_rows; ++q)
        if (const int i = bad_node(rho_pc + (size_t)q * N, N, true)) {
            set_error(where(fn, "rho_pc row", q) + "not finite or negative at node " + std::to_string(i));
            return DFTATOM_E_BAD_OPTION;
        }
    std::vector<int> dest_atom;
    std::vector<long long> dest_row;
    if (radial && (rc = batch_rows(*radial, orb_rows, dest_atom, dest_row))) return rc;
    const RadialDest rd{ radial, dest_atom.data(), dest_row.data(), true };
    const PseudoGroup pg{ v_ion, n_rows, atoms, any_core ? rho_pc : nullptr, any_core ? n_pc_rows : 0, pc_row };
    return solve_group(c, opts.data(), configs, n_atoms, out, steps, steps_stride, radial ? &rd : nullptr, &pg);
}

// ---------------------------------------------------------------------------------------------------------
// component entry points (host buffers)
// ---------------------------------------------------------------------------------------------------------

static int numerov_lanes_impl(dftatom_ctx* c, const double* V, int levels, double delta, double max_r, int n_lanes_in, const int* l_in,
                             const double* E_in, const int* limit_in, int impl, int* y0_sign_out, double* y0_log2_out, int* count_out,
                             int reps, float* ms_per_launch, double* node_steps)
{
    if (!c || !V || n_lanes_in <= 0 || !l_in || !E_in || !limit_in) return DFTATOM_E_ARG;
    // the production sweep shares one (potential, l) table tile per warp: group the lanes by l, pad every group to 32
    std::vector<int> perm, lv, limv; std::vector<double> Ev;
    for (int ll = 0; ll < 8; ++ll) {
        size_t before = lv.size();
        for (int k = 0; k < n_lanes_in; ++k) if (l_in[k] == ll) { perm.push_back(k); lv.push_back(ll); Ev.push_back(E_in[k]); limv.push_back(limit_in[k]); }
        while (lv.size() > before && (lv.size() & 31)) { perm.push_back(-1); lv.push_back(ll); Ev.push_back(Ev.back()); limv.push_back(limv.back()); }
    }
    if (lv.empty()) { set_error("l out of range"); return DFTATOM_E_ARG; }
    const int n_lanes = (int)lv.size();
    const int* l = lv.data(); const double* E = Ev.data(); const int* nodes_limit = limv.data();
    std::vector<int> hs(n_lanes), hc(n_lanes); std::vector<double> hl(n_lanes);
    int* y0_sign = hs.data(); double* y0_log2 = hl.data(); int* count = hc.data();
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    DevBuf& dV = c->scratch[0]; DevBuf& dA = c->scratch[1]; DevBuf& di = c->scratch[2]; DevBuf& dd = c->scratch[3];
    if ((rc = dV.ensure(sizeof(double) * N)) || (rc = dA.ensure(sizeof(double) * N))) return rc;
    if ((rc = di.ensure(sizeof(int) * (size_t)n_lanes * 5)) || (rc = dd.ensure(sizeof(double) * (size_t)n_lanes * 2))) return rc;
    DFT_CHECK(cudaMemcpyAsync(dV.p, V, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    launch_build_atab(g, dV.as<double>(), dA.as<double>(), 1, st);
    int* d_tab = di.as<int>(); int* d_l = d_tab + n_lanes; int* d_lim = d_l + n_lanes; int* d_sign = d_lim + n_lanes; int* d_cnt = d_sign + n_lanes;
    double* d_E = dd.as<double>(); double* d_log = d_E + n_lanes;
    DFT_CHECK(cudaMemsetAsync(d_tab, 0, sizeof(int) * n_lanes, st));
    DFT_CHECK(cudaMemcpyAsync(d_l, l, sizeof(int) * n_lanes, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(d_lim, nodes_limit, sizeof(int) * n_lanes, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(d_E, E, sizeof(double) * n_lanes, cudaMemcpyHostToDevice, st));
    NumerovLaneArgs a{ dA.as<double>(), n_lanes, d_tab, d_l, d_E, d_lim, d_sign, d_log, d_cnt };
    if (impl >= 4 && impl <= 6) launch_numerov_lanes_rows(g, a, 1 << (impl - 4), st); else if (impl == 0) launch_numerov_lanes_fast(g, a, st); else if (impl == 2) launch_numerov_lanes_seg(g, a, c->segments(N) > 1 ? c->segments(N) : 32, st); else if (impl == 3) launch_numerov_lanes_outward(g, a, st); else launch_numerov_lanes(g, a, st);
    if (reps > 0) {          // microbench: the same launch `reps` more times between CUDA events (tables and lanes resident)
        cudaEvent_t e0, e1;
        DFT_CHECK(cudaEventCreate(&e0)); DFT_CHECK(cudaEventCreate(&e1));
        DFT_CHECK(cudaEventRecord(e0, st));
        for (int r = 0; r < reps; ++r) { if (impl >= 4 && impl <= 6) launch_numerov_lanes_rows(g, a, 1 << (impl - 4), st); else if (impl == 0) launch_numerov_lanes_fast(g, a, st); else if (impl == 2) launch_numerov_lanes_seg(g, a, c->segments(N) > 1 ? c->segments(N) : 32, st); else if (impl == 3) launch_numerov_lanes_outward(g, a, st); else launch_numerov_lanes(g, a, st); }
        DFT_CHECK(cudaEventRecord(e1, st));
        DFT_CHECK(cudaStreamSynchronize(st));
        float ms = 0.f;
        DFT_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        if (ms_per_launch) *ms_per_launch = ms / (float)reps;
    }
    if (node_steps) {        // algorithmic work: (cut-off index - 1) node-steps per lane (Numerov.h:119-136, 1e-200 cut-off)
        double ns = 0.;
        for (int k = 0; k < n_lanes_in; ++k) {
            const double kappa = std::sqrt(2. * std::fabs(E_in[k]));
            int hi = N - 1, lo = 1;                         // same rule as numerov_common.cuh:start_index
            while (hi - lo > 1) {
                const int mid = (hi + lo) >> 1;
                const double arg = -(g.rp * std::expm1(delta * (double)mid)) * kappa - (double)mid * 0.5 * delta;
                if (arg < kFarLog) hi = mid; else lo = mid;
            }
            ns += (double)(hi - 1);
        }
        *node_steps = ns;
    }
    if (y0_sign) DFT_CHECK(cudaMemcpyAsync(y0_sign, d_sign, sizeof(int) * n_lanes, cudaMemcpyDeviceToHost, st));
    if (y0_log2) DFT_CHECK(cudaMemcpyAsync(y0_log2, d_log, sizeof(double) * n_lanes, cudaMemcpyDeviceToHost, st));
    if (count) DFT_CHECK(cudaMemcpyAsync(count, d_cnt, sizeof(int) * n_lanes, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    for (int k = 0; k < n_lanes; ++k) {
        if (perm[k] < 0) continue;
        if (y0_sign_out) y0_sign_out[perm[k]] = hs[k];
        if (y0_log2_out) y0_log2_out[perm[k]] = hl[k];
        if (count_out) count_out[perm[k]] = hc[k];
    }
    return 0;
}

int dftatom_numerov_lanes(dftatom_ctx* c, const double* V, int levels, double delta, double max_r, int n_lanes, const int* l,
                          const double* E, const int* nodes_limit, int impl, int* y0_sign, double* y0_log2, int* count)
{
    return numerov_lanes_impl(c, V, levels, delta, max_r, n_lanes, l, E, nodes_limit, impl, y0_sign, y0_log2, count, 0, nullptr, nullptr);
}

int dftatom_numerov_lanes_timed(dftatom_ctx* c, const double* V, int levels, double delta, double max_r, int n_lanes, const int* l,
                                const double* E, const int* nodes_limit, int impl, int* y0_sign, double* y0_log2, int* count,
                                int reps, float* ms_per_launch, double* lane_node_steps)
{
    if (reps <= 0) return DFTATOM_E_ARG;
    return numerov_lanes_impl(c, V, levels, delta, max_r, n_lanes, l, E, nodes_limit, impl, y0_sign, y0_log2, count, reps, ms_per_launch,
                              lane_node_steps);
}

static int poisson_cold(dftatom_ctx* c, const GridDev& g, int n_dens, const double* d_rho, const double* d_zbc, int* d_vcycles, long long* ld_out,
                        bool* streamed);

int dftatom_log_derivatives(dftatom_ctx* c, int levels, double delta, double max_r, const double* V, int n_pot, const int* pot, const int* l,
                            const double* r_c, int n_channels, const double* E, int n_energies, dftatom_logderiv* out, double* r_used)
{
    if (!c || !V || !pot || !l || !r_c || !E || !out) { set_error("dftatom_log_derivatives: NULL argument"); return DFTATOM_E_ARG; }
    if (n_pot < 1 || n_channels < 1 || n_energies < 1) { set_error("dftatom_log_derivatives: n_pot, n_channels and n_energies must be >= 1"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; GridEntry* ge; int rc = get_grid(c, levels, delta, max_r, &gp, &ge); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    if (N < 5) { set_error("dftatom_log_derivatives: the grid needs at least 5 nodes"); return DFTATOM_E_ARG; }
    static const char* const fn = "dftatom_log_derivatives";
    const std::vector<double>& r = ge->r;
    std::vector<int> ic(n_channels);
    for (int k = 0; k < n_channels; ++k) {
        const std::string at = where(fn, "channel", k);
        if (pot[k] < 0 || pot[k] >= n_pot) { set_error(at + "pot = " + std::to_string(pot[k]) + " outside 0.." + std::to_string(n_pot - 1)); return DFTATOM_E_ARG; }
        if (l[k] < 0 || l[k] > 3) { set_error(at + "l = " + std::to_string(l[k]) + " outside 0..3"); return DFTATOM_E_ARG; }
        if ((ic[k] = radius_node(r, r_c[k], 2, at, "r_c")) < 0) return DFTATOM_E_ARG;
    }
    for (int k = 0; k < n_energies; ++k)
        if (!std::isfinite(E[k])) { set_error(where(fn, "energy", k) + "E is not finite"); return DFTATOM_E_ARG; }
    for (int p = 0; p < n_pot; ++p)
        if (const int i = bad_node(V + (size_t)p * N, N)) { set_error(where(fn, "potential row", p) + "V is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    const int eb = (n_energies + 31) / 32;
    const long long n_warps_ll = (long long)n_channels * eb;
    if (n_warps_ll > (1LL << 30)) { set_error("dftatom_log_derivatives: too many (channel, energy) lanes"); return DFTATOM_E_ARG; }
    const int n_warps = (int)n_warps_ll;
    std::vector<int> h_int(pot, pot + n_channels);                  // pot | l | ic | warp_item
    h_int.insert(h_int.end(), l, l + n_channels);
    h_int.insert(h_int.end(), ic.begin(), ic.end());
    const std::vector<int> wi = warp_order(std::vector<long long>(ic.begin(), ic.end()), eb);
    h_int.insert(h_int.end(), wi.begin(), wi.end());
    DevBuf& dV = c->scratch[0]; DevBuf& dA = c->scratch[1]; DevBuf& di = c->scratch[2]; DevBuf& dd = c->scratch[3]; DevBuf& dO = c->scratch[4];
    const size_t nV = (size_t)n_pot * N, n_out = (size_t)n_channels * n_energies;
    if ((rc = dV.ensure(sizeof(double) * nV)) || (rc = dA.ensure(sizeof(double) * nV)) || (rc = di.ensure(sizeof(int) * h_int.size())) ||
        (rc = dd.ensure(sizeof(double) * n_energies)) || (rc = dO.ensure(sizeof(dftatom_logderiv) * n_out))) return rc;
    DFT_CHECK(cudaMemcpyAsync(dV.p, V, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(di.p, h_int.data(), sizeof(int) * h_int.size(), cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dd.p, E, sizeof(double) * n_energies, cudaMemcpyHostToDevice, st));
    launch_build_atab(g, dV.as<double>(), dA.as<double>(), n_pot, st);
    const int* d_i = di.as<int>();
    LogDerivArgs a{ dA.as<double>(), d_i, d_i + n_channels, d_i + 2 * (size_t)n_channels, dd.as<double>(), n_energies,
                    d_i + 3 * (size_t)n_channels, n_warps, eb, dO.as<dftatom_logderiv>() };
    launch_logderiv(g, a, st);
    DFT_CHECK(cudaGetLastError());
    DFT_CHECK(cudaMemcpyAsync(out, dO.p, sizeof(dftatom_logderiv) * n_out, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    if (r_used) for (int k = 0; k < n_channels; ++k) r_used[k] = r[ic[k]];
    return 0;
}

int dftatom_grid_nodes(dftatom_ctx* c, int levels, double delta, double max_r, double* r)
{
    if (!c || !r) { set_error("dftatom_grid_nodes: NULL argument"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; GridEntry* ge; int rc = get_grid(c, levels, delta, max_r, &gp, &ge); if (rc) return rc;
    std::copy(ge->r.begin(), ge->r.end(), r);
    return 0;
}

int dftatom_tm_pseudize(dftatom_ctx* c, int levels, double delta, double max_r, const double* V, int n_pot, const double* u, int n_orb,
                        const dftatom_tm_channel* ch, int n_channels, dftatom_tm_result* out, double* u_ps, double* v_scr,
                        double* v_ion, double* rho_val)
{
    return dftatom_tm_pseudize_core(c, levels, delta, max_r, V, n_pot, u, n_orb, ch, n_channels, out, u_ps, v_scr, v_ion, rho_val, nullptr);
}

int dftatom_tm_pseudize_core(dftatom_ctx* c, int levels, double delta, double max_r, const double* V, int n_pot, const double* u, int n_orb,
                             const dftatom_tm_channel* ch, int n_channels, dftatom_tm_result* out, double* u_ps, double* v_scr,
                             double* v_ion, double* rho_val, const double* rho_pc)
{
    if (!c || !V || !u || !ch || !out) { set_error("dftatom_tm_pseudize: NULL argument"); return DFTATOM_E_ARG; }
    if (n_pot < 1 || n_orb < 1 || n_channels < 1) { set_error("dftatom_tm_pseudize: n_pot, n_orb and n_channels must be >= 1"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; GridEntry* ge; int rc = get_grid(c, levels, delta, max_r, &gp, &ge); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    if (N < 7) { set_error("dftatom_tm_pseudize: the grid needs at least 7 nodes"); return DFTATOM_E_ARG; }
    if ((long long)n_channels + n_pot > 65535 || (long long)std::max(n_pot, n_channels) * N >= (1LL << 31)) {
        set_error("dftatom_tm_pseudize: too many channels or potential rows for one call"); return DFTATOM_E_ARG;
    }
    static const char* const fn = "dftatom_tm_pseudize";
    const std::vector<double>& r = ge->r;
    for (int p = 0; p < n_pot; ++p)
        if (const int i = bad_node(V + (size_t)p * N, N)) { set_error(where(fn, "potential row", p) + "V is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    for (int o = 0; o < n_orb; ++o)
        if (const int i = bad_node(u + (size_t)o * N, N)) { set_error(where(fn, "orbital row", o) + "u is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    for (int p = 0; rho_pc && p < n_pot; ++p)
        if (const int i = bad_node(rho_pc + (size_t)p * N, N, true)) { set_error(where(fn, "rho_pc row", p) + "not finite or negative at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    std::vector<int> ic(n_channels);
    std::vector<unsigned> l_taken(n_pot, 0u);             // per potential row: bit l set once a channel takes l
    for (int k = 0; k < n_channels; ++k) {
        const dftatom_tm_channel& q = ch[k];
        const std::string at = where(fn, "channel", k);
        if (q.pot < 0 || q.pot >= n_pot) { set_error(at + "pot = " + std::to_string(q.pot) + " outside 0.." + std::to_string(n_pot - 1)); return DFTATOM_E_ARG; }
        if (q.orbital < 0 || q.orbital >= n_orb) { set_error(at + "orbital = " + std::to_string(q.orbital) + " outside 0.." + std::to_string(n_orb - 1)); return DFTATOM_E_ARG; }
        if (q.l < 0 || q.l > 3) { set_error(at + "l = " + std::to_string(q.l) + " outside 0..3"); return DFTATOM_E_ARG; }
        if (l_taken[q.pot] & (1u << q.l)) { set_error(at + "l = " + std::to_string(q.l) + " already taken by another channel of potential row " + std::to_string(q.pot)); return DFTATOM_E_ARG; }
        l_taken[q.pot] |= 1u << q.l;
        if ((ic[k] = radius_node(r, q.r_c, 3, at, "r_c")) < 0) return DFTATOM_E_ARG;      // i_c >= 3: the 5-point stencil of V' and V'' stays off node 0
        if (!std::isfinite(q.eps)) { set_error(at + "eps is not finite"); return DFTATOM_E_ARG; }
        if (!(q.occ >= 0. && q.occ <= 2. * (2 * q.l + 1))) { set_error(at + "occ is not finite or outside [0, 2(2l+1)]"); return DFTATOM_E_ARG; }
        const double* ur = u + (size_t)q.orbital * N;
        if (ur[ic[k]] == 0.) { set_error(at + "u is 0 at r_c (node " + std::to_string(ic[k]) + ")"); return DFTATOM_E_ARG; }
        const bool pos = ur[ic[k]] > 0.;
        for (int i = ic[k] + 1; i < N; ++i)
            if (pos ? ur[i] < 0. : ur[i] > 0.) { set_error(at + "u changes sign at node " + std::to_string(i) + " beyond r_c: r_c lies inside the outermost node"); return DFTATOM_E_ARG; }
    }
    // host tables: the channels dealt longest i_c first; the channels of each potential row; rows with electrons first (their Poisson solves)
    std::vector<int> order(n_channels);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return ic[a] > ic[b]; });
    std::vector<int> row_begin(n_pot + 1, 0), row_chan(n_channels), slot(n_pot);
    std::vector<double> qv(n_pot, 0.), eps(n_channels), occ(n_channels);
    for (int k = 0; k < n_channels; ++k) { ++row_begin[ch[k].pot + 1]; qv[ch[k].pot] += ch[k].occ; eps[k] = ch[k].eps; occ[k] = ch[k].occ; }
    for (int p = 0; p < n_pot; ++p) row_begin[p + 1] += row_begin[p];
    {
        std::vector<int> fill(row_begin.begin(), row_begin.end() - 1);
        for (int k = 0; k < n_channels; ++k) row_chan[fill[ch[k].pot]++] = k;
    }
    int n_solve = 0;
    for (int p = 0; p < n_pot; ++p) if (qv[p] > 0.) slot[p] = n_solve++;
    std::vector<double> zbc;
    for (int p = 0; p < n_pot; ++p) if (qv[p] > 0.) zbc.push_back(qv[p]);
    for (int p = 0, s = n_solve; p < n_pot; ++p) if (!(qv[p] > 0.)) slot[p] = s++;
    std::vector<int> h_int;                                   // pot | orbital | l | ic | order | row_chan | row_begin | slot
    for (int k = 0; k < n_channels; ++k) h_int.push_back(ch[k].pot);
    for (int k = 0; k < n_channels; ++k) h_int.push_back(ch[k].orbital);
    for (int k = 0; k < n_channels; ++k) h_int.push_back(ch[k].l);
    h_int.insert(h_int.end(), ic.begin(), ic.end());
    h_int.insert(h_int.end(), order.begin(), order.end());
    h_int.insert(h_int.end(), row_chan.begin(), row_chan.end());
    h_int.insert(h_int.end(), row_begin.begin(), row_begin.end());
    h_int.insert(h_int.end(), slot.begin(), slot.end());
    std::vector<double> h_dbl(eps);                           // eps | occ | zbc
    h_dbl.insert(h_dbl.end(), occ.begin(), occ.end());
    h_dbl.insert(h_dbl.end(), zbc.begin(), zbc.end());
    const size_t nV = (size_t)n_pot * N, nU = (size_t)n_orb * N, nC = (size_t)n_channels * N;
    DevBuf& dD = c->scratch[0]; DevBuf& dI = c->scratch[1]; DevBuf& dR = c->scratch[2]; DevBuf& dv = c->scratch[3];
    const size_t n_dbl = 6 * nV + nU + 3 * nC + h_dbl.size() + (rho_pc ? 2 * nV : 0);      // V atab rho rho_out vxc edif | u | u_ps v_scr v_ion | eps occ zbc | rho_pc rho_xc
    if ((rc = dD.ensure(sizeof(double) * n_dbl)) || (rc = dI.ensure(sizeof(int) * h_int.size())) || (rc = dR.ensure(sizeof(dftatom_tm_result) * n_channels)) ||
        (rc = dv.ensure(sizeof(int) * n_pot))) return rc;
    double* d = dD.as<double>();
    double* dV = d; double* dA = dV + nV; double* drho = dA + nV; double* drho_out = drho + nV; double* dvxc = drho_out + nV; double* dedif = dvxc + nV;
    double* du = dedif + nV; double* dups = du + nU; double* dvscr = dups + nC; double* dvion = dvscr + nC; double* dh = dvion + nC;
    const int* di = dI.as<int>();
    DFT_CHECK(cudaMemcpyAsync(dV, V, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(du, u, sizeof(double) * nU, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dh, h_dbl.data(), sizeof(double) * h_dbl.size(), cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dI.p, h_int.data(), sizeof(int) * h_int.size(), cudaMemcpyHostToDevice, st));
    double* dpc = dh + h_dbl.size(); double* dxc = dpc + nV;
    if (rho_pc) DFT_CHECK(cudaMemcpyAsync(dpc, rho_pc, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    launch_build_atab(g, dV, dA, n_pot, st);
    const size_t nc = (size_t)n_channels;
    TmArgs ta{ dV, dA, du, di, di + nc, di + 2 * nc, di + 3 * nc, dh, di + 4 * nc, n_channels, dR.as<dftatom_tm_result>(), dups, dvscr };
    launch_tm(g, ta, st);
    TmRowArgs ra{ n_pot, n_channels, di + 6 * nc, di + 5 * nc, di, dh + nc, dR.as<dftatom_tm_result>(), dups, dvscr, di + 6 * nc + n_pot + 1, n_solve,
                  drho, nullptr, N, dvxc, dvion, drho_out };
    launch_tm_density(g, ra, st);
    if (n_solve > 0) {
        long long ld = N; bool streamed = false;
        if ((rc = poisson_cold(c, g, n_solve, drho, dh + 2 * nc, dv.as<int>(), &ld, &streamed))) return rc;
        ra.U = c->ubuf.as<double>(); ra.ldU = ld;
    }
    if (rho_pc) {           // V_xc of rho_val + rho_pc; V_H and rho_out keep reading rho_val
        launch_core_xc_density(g, n_pot, di + 6 * nc + n_pot + 1, drho, dpc, dxc, st);
        launch_vwn((int)nV, dxc, nullptr, nullptr, nullptr, dvxc, dedif, st);
    } else {
        launch_vwn((int)nV, drho, nullptr, nullptr, nullptr, dvxc, dedif, st);
    }
    launch_tm_unscreen(g, ra, st);
    DFT_CHECK(cudaGetLastError());
    DFT_CHECK(cudaMemcpyAsync(out, dR.p, sizeof(dftatom_tm_result) * n_channels, cudaMemcpyDeviceToHost, st));
    if (u_ps) DFT_CHECK(cudaMemcpyAsync(u_ps, dups, sizeof(double) * nC, cudaMemcpyDeviceToHost, st));
    if (v_scr) DFT_CHECK(cudaMemcpyAsync(v_scr, dvscr, sizeof(double) * nC, cudaMemcpyDeviceToHost, st));
    if (v_ion) DFT_CHECK(cudaMemcpyAsync(v_ion, dvion, sizeof(double) * nC, cudaMemcpyDeviceToHost, st));
    if (rho_val) DFT_CHECK(cudaMemcpyAsync(rho_val, drho_out, sizeof(double) * nV, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_partial_core(dftatom_ctx* c, int levels, double delta, double max_r, const double* u, int n_orb, const dftatom_core_orbital* core,
                         int n_core, const double* r_pc, int n_rows, dftatom_pcc_result* out, double* rho_core, double* rho_pc)
{
    if (!c || !u || !r_pc || !out || (n_core > 0 && !core)) { set_error("dftatom_partial_core: NULL argument"); return DFTATOM_E_ARG; }
    if (n_orb < 1 || n_rows < 1 || n_core < 0) { set_error("dftatom_partial_core: n_orb and n_rows must be >= 1, n_core >= 0"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; GridEntry* ge; int rc = get_grid(c, levels, delta, max_r, &gp, &ge); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    if (N < 7) { set_error("dftatom_partial_core: the grid needs at least 7 nodes"); return DFTATOM_E_ARG; }
    if (n_rows > 65535 || (long long)std::max(n_rows, n_orb) * N >= (1LL << 31)) { set_error("dftatom_partial_core: too many rows for one call"); return DFTATOM_E_ARG; }
    static const char* const fn = "dftatom_partial_core";
    std::vector<int> ipc(n_rows, 0);
    for (int p = 0; p < n_rows; ++p)       // r_pc = 0: the full core
        if (r_pc[p] != 0. && (ipc[p] = radius_node(ge->r, r_pc[p], 3, where(fn, "row", p), "r_pc")) < 0) return DFTATOM_E_ARG;
    std::vector<int> begin(n_rows + 1, 0), orb(n_core);
    std::vector<double> occ(n_core);
    for (int k = 0; k < n_core; ++k) {
        const dftatom_core_orbital& e = core[k];
        const std::string at = where(fn, "core entry", k);
        if (e.row < 0 || e.row >= n_rows) { set_error(at + "row = " + std::to_string(e.row) + " outside 0.." + std::to_string(n_rows - 1)); return DFTATOM_E_ARG; }
        if (e.orbital < 0 || e.orbital >= n_orb) { set_error(at + "orbital = " + std::to_string(e.orbital) + " outside 0.." + std::to_string(n_orb - 1)); return DFTATOM_E_ARG; }
        if (!(e.occ >= 0. && e.occ <= 14.)) { set_error(at + "occ is not finite or outside [0, 14]"); return DFTATOM_E_ARG; }
        ++begin[e.row + 1];
    }
    for (int o = 0; o < n_orb; ++o)
        if (const int i = bad_node(u + (size_t)o * N, N)) { set_error(where(fn, "orbital row", o) + "u is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    for (int p = 0; p < n_rows; ++p) begin[p + 1] += begin[p];
    {
        std::vector<int> fill(begin.begin(), begin.end() - 1);
        for (int k = 0; k < n_core; ++k) { const int q = fill[core[k].row]++; orb[q] = core[k].orbital; occ[q] = core[k].occ; }
    }
    std::vector<int> h_int(begin);                               // core_begin | core_orb | ipc
    h_int.insert(h_int.end(), orb.begin(), orb.end());
    h_int.insert(h_int.end(), ipc.begin(), ipc.end());
    const size_t nU = (size_t)n_orb * N, nR = (size_t)n_rows * N;
    DevBuf& dD = c->scratch[0]; DevBuf& dI = c->scratch[1]; DevBuf& dR = c->scratch[2];
    if ((rc = dD.ensure(sizeof(double) * (nU + 2 * nR + std::max(n_core, 1)))) || (rc = dI.ensure(sizeof(int) * h_int.size())) ||
        (rc = dR.ensure(sizeof(dftatom_pcc_result) * n_rows))) return rc;
    double* du = dD.as<double>(); double* dcore = du + nU; double* dpc = dcore + nR; double* docc = dpc + nR;
    DFT_CHECK(cudaMemcpyAsync(du, u, sizeof(double) * nU, cudaMemcpyHostToDevice, st));
    if (n_core) DFT_CHECK(cudaMemcpyAsync(docc, occ.data(), sizeof(double) * n_core, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dI.p, h_int.data(), sizeof(int) * h_int.size(), cudaMemcpyHostToDevice, st));
    const int* di = dI.as<int>();
    PcArgs pa{ du, di, di + n_rows + 1, docc, di + n_rows + 1 + n_core, n_rows, dR.as<dftatom_pcc_result>(), dcore, dpc };
    launch_partial_core(g, pa, st);
    DFT_CHECK(cudaGetLastError());
    DFT_CHECK(cudaMemcpyAsync(out, dR.p, sizeof(dftatom_pcc_result) * n_rows, cudaMemcpyDeviceToHost, st));
    if (rho_core) DFT_CHECK(cudaMemcpyAsync(rho_core, dcore, sizeof(double) * nR, cudaMemcpyDeviceToHost, st));
    if (rho_pc) DFT_CHECK(cudaMemcpyAsync(rho_pc, dpc, sizeof(double) * nR, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

// shared by level_search / numerov_orbital / kb_form: n_rows pseudo-atoms, atom k with potential row k (V[n_rows][N]) and nuclear charge
// Z[k] (which sets its search bracket [-Z^2 - 1, 50])
static int setup_rows(dftatom_ctx* c, const GridDev& g, const double* V, int n_rows, const int* Z, const std::vector<OrbitalDev>& orbs,
                      AtomDev** d_atoms, AtomState** d_astate, OrbitalDev** d_orbs, SearchState** d_ss, double** d_atab)
{
    const size_t nV = (size_t)n_rows * g.N; cudaStream_t st = c->stream;
    int rc;
    DevBuf& dV = c->scratch[0]; DevBuf& dA = c->scratch[1];
    if ((rc = dV.ensure(sizeof(double) * nV)) || (rc = dA.ensure(sizeof(double) * nV))) return rc;
    DFT_CHECK(cudaMemcpyAsync(dV.p, V, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    launch_build_atab(g, dV.as<double>(), dA.as<double>(), n_rows, st);
    std::vector<AtomDev> atoms(n_rows);
    for (int k = 0; k < n_rows; ++k) { atoms[k] = AtomDev{}; atoms[k].Z = Z[k]; atoms[k].n_spin = 1; }
    std::vector<AtomState> as(n_rows, AtomState{ 0., 0, 0, 0, 0 });
    if ((rc = upload(c, c->scratch[4], atoms)) || (rc = upload(c, c->scratch[5], as)) || (rc = upload(c, c->scratch[6], orbs))) return rc;
    if ((rc = c->scratch[7].ensure(sizeof(SearchState) * orbs.size()))) return rc;
    *d_atoms = c->scratch[4].as<AtomDev>(); *d_astate = c->scratch[5].as<AtomState>(); *d_orbs = c->scratch[6].as<OrbitalDev>();
    *d_ss = c->scratch[7].as<SearchState>(); *d_atab = dA.as<double>();
    return 0;
}

// the production energy search of every orbital (OrbitalDev.atom = .tab = its potential row) on the rows V[n_rows][N]; E_out / converged_out
// (may be NULL) as dftatom_level_search returns them
static int search_levels(dftatom_ctx* c, const GridDev& g, const double* V, int n_rows, const int* Z, const std::vector<OrbitalDev>& orbs,
                         double* E_out, int* converged_out)
{
    const int n_levels = (int)orbs.size(); cudaStream_t st = c->stream;
    AtomDev* da; AtomState* ds; OrbitalDev* dorb; SearchState* dss; double* datab;
    int rc;
    if ((rc = setup_rows(c, g, V, n_rows, Z, orbs, &da, &ds, &dorb, &dss, &datab))) return rc;
    launch_search_init(g, da, ds, dorb, dss, n_levels, st);
    const int rounds = search_rounds_needed(*std::max_element(Z, Z + n_rows));
    if (c->k.search_mode == 0 && c->k.search_kernel == 0 && !g.uniform) launch_search_rows(g, datab, da, dorb, ds, dss, n_levels, nullptr, 0, c->k.rows_cfg, 0, 0, 1 << 30, st);
    else if (c->k.search_mode == 0 && c->segments(g.N) > 1) launch_search_seg(g, datab, da, dorb, ds, dss, n_levels, nullptr, c->segments(g.N), nullptr, 0, 0, st);
    else if (c->k.search_mode == 0) launch_search_fused(g, datab, da, dorb, ds, dss, n_levels, nullptr, nullptr, 0, 0, st);
    else for (int r = 0; r < rounds; ++r) launch_search_round(g, datab, dorb, ds, dss, n_levels, nullptr, st);
    std::vector<SearchState> h(n_levels);
    DFT_CHECK(cudaMemcpyAsync(h.data(), dss, sizeof(SearchState) * n_levels, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    for (int k = 0; k < n_levels; ++k) {
        const bool fin = h[k].stage == 3;
        if (E_out) E_out[k] = fin ? h[k].E : (h[k].stage == 0 ? h[k].dn_hi : h[k].bot);
        if (converged_out) converged_out[k] = fin ? h[k].converged : 0;
    }
    return 0;
}

int dftatom_level_search(dftatom_ctx* c, const double* V, int levels, double delta, double max_r, int Z, int n_levels,
                         const int* n, const int* l, double* E_out, int* converged_out)
{
    if (!c || !V || n_levels <= 0) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp;
    std::vector<OrbitalDev> orbs(n_levels);
    for (int k = 0; k < n_levels; ++k) { orbs[k] = OrbitalDev{ 0, 0, n[k] - 1, l[k], 1, n[k] - 1 - l[k], 0 }; }
    return search_levels(c, g, V, 1, &Z, orbs, E_out, converged_out);
}

int dftatom_kb_form(dftatom_ctx* c, int levels, double delta, double max_r, const double* V, const double* u, int n_rows,
                    const dftatom_kb_channel* ch, int n_channels, dftatom_kb_result* out, double* beta)
{
    if (!c || !V || !u || !ch || !out) { set_error("dftatom_kb_form: NULL argument"); return DFTATOM_E_ARG; }
    if (n_rows < 1 || n_channels < 1) { set_error("dftatom_kb_form: n_rows and n_channels must be >= 1"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    if (N < 7) { set_error("dftatom_kb_form: the grid needs at least 7 nodes"); return DFTATOM_E_ARG; }
    if (n_channels > 65535 || (long long)std::max(n_rows, n_channels) * N >= (1LL << 31)) {
        set_error("dftatom_kb_form: too many channels or rows for one call"); return DFTATOM_E_ARG;
    }
    static const char* const fn = "dftatom_kb_form";
    for (int p = 0; p < n_rows; ++p) {
        if (const int i = bad_node(V + (size_t)p * N, N)) { set_error(where(fn, "row", p) + "V is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
        if (const int i = bad_node(u + (size_t)p * N, N)) { set_error(where(fn, "row", p) + "u is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    }
    // i_s per channel, the search bracket of every local row, and the (loc, l) searches of the non-local channels (each searched once)
    std::vector<int> is(n_channels, 0), zb(n_rows, 0), srow_of(n_rows, -1), search_of(n_channels, -1), srows;
    std::map<std::pair<int, int>, int> searches;
    std::vector<OrbitalDev> orbs;
    for (int k = 0; k < n_channels; ++k) {
        const dftatom_kb_channel& q = ch[k];
        const std::string at = where(fn, "channel", k);
        if (q.row < 0 || q.row >= n_rows) { set_error(at + "row = " + std::to_string(q.row) + " outside 0.." + std::to_string(n_rows - 1)); return DFTATOM_E_ARG; }
        if (q.loc < 0 || q.loc >= n_rows) { set_error(at + "loc = " + std::to_string(q.loc) + " outside 0.." + std::to_string(n_rows - 1)); return DFTATOM_E_ARG; }
        if (q.l < 0 || q.l > 3) { set_error(at + "l = " + std::to_string(q.l) + " outside 0..3"); return DFTATOM_E_ARG; }
        if (!std::isfinite(q.eps)) { set_error(at + "eps is not finite"); return DFTATOM_E_ARG; }
        if (q.row == q.loc) continue;
        const double* a = V + (size_t)q.row * N; const double* b = V + (size_t)q.loc * N;
        for (int i = N - 1; i >= 1 && !is[k]; --i) if (a[i] != b[i]) is[k] = i;
        if (is[k] > N - 3) { set_error(at + "V[row] differs from V[loc] at node " + std::to_string(is[k]) + " > N - 3"); return DFTATOM_E_ARG; }
        if (!zb[q.loc]) {
            double vmin = b[1];
            for (int i = 2; i < N; ++i) vmin = std::min(vmin, b[i]);
            if (!(zb[q.loc] = bracket_z(vmin, 0.))) { set_error(at + "local potential too deep (min V[loc] = " + std::to_string(vmin) + " below -118^2 - 1)"); return DFTATOM_E_ARG; }
        }
        if (srow_of[q.loc] < 0) { srow_of[q.loc] = (int)srows.size(); srows.push_back(q.loc); }
        const auto key = std::make_pair(q.loc, q.l);
        auto it = searches.find(key);
        if (it == searches.end()) {
            it = searches.emplace(key, (int)orbs.size() / 2).first;
            const int sr = srow_of[q.loc];
            for (int w = 0; w < 2; ++w) orbs.push_back(OrbitalDev{ sr, 0, q.l + w, q.l, 1, w, sr });
        }
        search_of[k] = it->second;
    }
    std::vector<double> eloc(orbs.size(), NAN);
    std::vector<int> conv(orbs.size(), 0);
    if (!orbs.empty()) {
        std::vector<double> vs(srows.size() * (size_t)N);
        std::vector<int> zs(srows.size());
        for (size_t k = 0; k < srows.size(); ++k) { std::copy(V + (size_t)srows[k] * N, V + (size_t)(srows[k] + 1) * N, vs.begin() + k * N); zs[k] = zb[srows[k]]; }
        if ((rc = search_levels(c, g, vs.data(), (int)srows.size(), zs.data(), orbs, eloc.data(), conv.data()))) return rc;
    }
    std::vector<int> h_int(3 * (size_t)n_channels);                // row | loc | is
    for (int k = 0; k < n_channels; ++k) { h_int[k] = ch[k].row; h_int[n_channels + k] = ch[k].loc; h_int[2 * n_channels + k] = is[k]; }
    const size_t nV = (size_t)n_rows * N, nB = (size_t)n_channels * N;
    DevBuf& dD = c->scratch[0]; DevBuf& dI = c->scratch[1]; DevBuf& dR = c->scratch[2];
    if ((rc = dD.ensure(sizeof(double) * (2 * nV + nB))) || (rc = dI.ensure(sizeof(int) * h_int.size())) ||
        (rc = dR.ensure(sizeof(dftatom_kb_result) * n_channels))) return rc;
    double* dV = dD.as<double>(); double* du = dV + nV; double* dB = du + nV;
    DFT_CHECK(cudaMemcpyAsync(dV, V, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(du, u, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dI.p, h_int.data(), sizeof(int) * h_int.size(), cudaMemcpyHostToDevice, st));
    const int* di = dI.as<int>();
    KbFormArgs ka{ dV, du, di, di + n_channels, di + 2 * (size_t)n_channels, n_channels, dR.as<dftatom_kb_result>(), dB };
    launch_kb_form(g, ka, st);
    DFT_CHECK(cudaGetLastError());
    std::vector<dftatom_kb_result> res(n_channels);
    DFT_CHECK(cudaMemcpyAsync(res.data(), dR.p, sizeof(dftatom_kb_result) * n_channels, cudaMemcpyDeviceToHost, st));
    if (beta) DFT_CHECK(cudaMemcpyAsync(beta, dB, sizeof(double) * nB, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    // the GSS verdict (nodeless reference state): a ghost below eps iff eps lies above the local level with 1 node (E_KB > 0) or 0 nodes (E_KB < 0)
    for (int k = 0; k < n_channels; ++k) {
        dftatom_kb_result& r = res[k];
        r.pad = 0;
        if (r.status == 1) { r.eps_loc[0] = r.eps_loc[1] = NAN; r.ghost = 0; continue; }
        const int s = search_of[k];
        r.eps_loc[0] = eloc[2 * s]; r.eps_loc[1] = eloc[2 * s + 1];
        if (r.status == 0 && !(conv[2 * s] && conv[2 * s + 1])) r.status = 3;
        if (r.status != 0) { r.ghost = -1; continue; }
        r.ghost = r.E_KB > 0. ? (ch[k].eps > r.eps_loc[1]) : (ch[k].eps > r.eps_loc[0]);
    }
    std::copy(res.begin(), res.end(), out);
    return 0;
}

int dftatom_kb_log_derivatives(dftatom_ctx* c, int levels, double delta, double max_r, const double* V_loc, int n_pot,
                               const double* beta, int n_proj, const dftatom_kb_ld_channel* ch, int n_channels,
                               const double* E, int n_energies, dftatom_logderiv* out, double* r_used)
{
    if (!c || !V_loc || !ch || !E || !out || (n_proj > 0 && !beta)) { set_error("dftatom_kb_log_derivatives: NULL argument"); return DFTATOM_E_ARG; }
    if (n_pot < 1 || n_channels < 1 || n_energies < 1 || n_proj < 0) {
        set_error("dftatom_kb_log_derivatives: n_pot, n_channels and n_energies must be >= 1, n_proj >= 0"); return DFTATOM_E_ARG;
    }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; GridEntry* ge; int rc = get_grid(c, levels, delta, max_r, &gp, &ge); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    if (N < 5) { set_error("dftatom_kb_log_derivatives: the grid needs at least 5 nodes"); return DFTATOM_E_ARG; }
    if (n_proj > 65535) { set_error("dftatom_kb_log_derivatives: too many projectors for one call"); return DFTATOM_E_ARG; }
    static const char* const fn = "dftatom_kb_log_derivatives";
    const std::vector<double>& r = ge->r;
    std::vector<int> ic(n_channels), is(std::max(n_proj, 1), 0);
    for (int p = 0; p < n_proj; ++p) {
        const double* b = beta + (size_t)p * N;
        const int bad = std::isfinite(b[0]) ? bad_node(b, N) : 0;      // (beta is checked from node 0 on)
        if (bad || !std::isfinite(b[0])) { set_error(where(fn, "projector", p) + "beta is not finite at node " + std::to_string(bad)); return DFTATOM_E_ARG; }
        for (int i = 0; i < N; ++i) if (b[i] != 0.) is[p] = i;
        if (is[p] > N - 3) { set_error(where(fn, "projector", p) + "beta is not 0 at node " + std::to_string(is[p]) + " > N - 3"); return DFTATOM_E_ARG; }
    }
    for (int k = 0; k < n_channels; ++k) {
        const dftatom_kb_ld_channel& q = ch[k];
        const std::string at = where(fn, "channel", k);
        if (q.pot < 0 || q.pot >= n_pot) { set_error(at + "pot = " + std::to_string(q.pot) + " outside 0.." + std::to_string(n_pot - 1)); return DFTATOM_E_ARG; }
        if (q.proj < -1 || q.proj >= n_proj) { set_error(at + "proj = " + std::to_string(q.proj) + " outside -1.." + std::to_string(n_proj - 1)); return DFTATOM_E_ARG; }
        if (q.l < 0 || q.l > 3) { set_error(at + "l = " + std::to_string(q.l) + " outside 0..3"); return DFTATOM_E_ARG; }
        if (!std::isfinite(q.E_KB)) { set_error(at + "E_KB is not finite"); return DFTATOM_E_ARG; }
        if ((ic[k] = radius_node(r, q.r_c, 2, at, "r_c")) < 0) return DFTATOM_E_ARG;
    }
    for (int k = 0; k < n_energies; ++k)
        if (!std::isfinite(E[k])) { set_error(where(fn, "energy", k) + "E is not finite"); return DFTATOM_E_ARG; }
    for (int p = 0; p < n_pot; ++p)
        if (const int i = bad_node(V_loc + (size_t)p * N, N)) { set_error(where(fn, "potential row", p) + "V is not finite at node " + std::to_string(i)); return DFTATOM_E_ARG; }
    const int eb = (n_energies + 31) / 32;
    const long long n_warps_ll = (long long)n_channels * eb;
    if (n_warps_ll > (1LL << 30)) { set_error("dftatom_kb_log_derivatives: too many (channel, energy) lanes"); return DFTATOM_E_ARG; }
    const int n_warps = (int)n_warps_ll;
    // a channel with a projector sweeps to max(i_c, i_s) + 1 and again to i_c
    std::vector<long long> cost(n_channels);
    for (int k = 0; k < n_channels; ++k) cost[k] = ch[k].proj < 0 ? ic[k] : (long long)std::max(ic[k], is[ch[k].proj]) + ic[k];
    const size_t nc = (size_t)n_channels, np = (size_t)std::max(n_proj, 1);
    std::vector<int> h_int(4 * nc + np);                        // pot | l | ic | proj | is | warp_item
    for (size_t k = 0; k < nc; ++k) { h_int[k] = ch[k].pot; h_int[nc + k] = ch[k].l; h_int[2 * nc + k] = ic[k]; h_int[3 * nc + k] = ch[k].proj; }
    std::copy(is.begin(), is.end(), h_int.begin() + 4 * nc);
    const std::vector<int> wi = warp_order(cost, eb);
    h_int.insert(h_int.end(), wi.begin(), wi.end());
    std::vector<double> h_dbl(E, E + n_energies);                // E | E_KB
    for (int k = 0; k < n_channels; ++k) h_dbl.push_back(ch[k].E_KB);
    const size_t nV = (size_t)n_pot * N, nP = (size_t)n_proj * N, n_out = nc * n_energies;
    DevBuf& dD = c->scratch[0]; DevBuf& dI = c->scratch[1]; DevBuf& dO = c->scratch[2];
    if ((rc = dD.ensure(sizeof(double) * (2 * nV + 3 * nP + h_dbl.size()))) || (rc = dI.ensure(sizeof(int) * h_int.size())) ||
        (rc = dO.ensure(sizeof(dftatom_logderiv) * n_out))) return rc;
    double* dV = dD.as<double>(); double* dA = dV + nV; double* dB = dA + nV; double* dS = dB + nP; double* dH = dS + nP; double* dE = dH + nP;
    DFT_CHECK(cudaMemcpyAsync(dV, V_loc, sizeof(double) * nV, cudaMemcpyHostToDevice, st));
    if (n_proj > 0) DFT_CHECK(cudaMemcpyAsync(dB, beta, sizeof(double) * nP, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dE, h_dbl.data(), sizeof(double) * h_dbl.size(), cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dI.p, h_int.data(), sizeof(int) * h_int.size(), cudaMemcpyHostToDevice, st));
    launch_build_atab(g, dV, dA, n_pot, st);
    const int* d_i = dI.as<int>();
    if (n_proj > 0) launch_kb_proj(g, KbProjArgs{ dB, d_i + 4 * nc, n_proj, dS, dH }, st);
    KbLogDerivArgs a{ dA, d_i, d_i + nc, d_i + 2 * nc, d_i + 3 * nc, dE + n_energies, dS, dH, d_i + 4 * nc, dE, n_energies,
                      d_i + 4 * nc + np, n_warps, eb, dO.as<dftatom_logderiv>() };
    launch_kb_logderiv(g, a, st);
    DFT_CHECK(cudaGetLastError());
    DFT_CHECK(cudaMemcpyAsync(out, dO.p, sizeof(dftatom_logderiv) * n_out, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    if (r_used) for (int k = 0; k < n_channels; ++k) r_used[k] = r[ic[k]];
    return 0;
}

int dftatom_numerov_orbital(dftatom_ctx* c, const double* V, int levels, double delta, double max_r, int l, double E,
                            double* u_out, int* match_point)
{
    if (!c || !V || !u_out) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    std::vector<OrbitalDev> orbs(1); orbs[0] = OrbitalDev{ 0, 0, l, l, 1, 0, 0 };
    AtomDev* da; AtomState* ds; OrbitalDev* dorb; SearchState* dss; double* datab;
    const int Z = 1;
    if ((rc = setup_rows(c, g, V, 1, &Z, orbs, &da, &ds, &dorb, &dss, &datab))) return rc;
    SearchState s{}; s.E = E; s.stage = 3; s.converged = 1;
    DFT_CHECK(cudaMemcpyAsync(dss, &s, sizeof(s), cudaMemcpyHostToDevice, st));
    // single-atom ScfBuffers so that density_update's normalisation path is the one exercised
    if ((rc = c->psi.ensure(sizeof(double) * N)) || (rc = c->match_pt.ensure(sizeof(int)))) return rc;
    if ((rc = c->inv_norm.ensure(sizeof(double)))) return rc;
    if (c->k.match_mode == 0) launch_match_cta(g, datab, dorb, ds, dss, c->psi.as<double>(), c->match_pt.as<int>(), c->inv_norm.as<double>(), 1, 0, 0, 0, 1 << 30, st);
    else if (c->k.match_mode == 2) launch_match_seg(g, datab, dorb, ds, dss, c->psi.as<double>(), c->match_pt.as<int>(), 1, st);
    else launch_match(g, datab, dorb, ds, dss, c->psi.as<double>(), c->match_pt.as<int>(), 1, st);
    std::vector<double> y(N), sq(N), wj(N);
    int mp = 0;
    DFT_CHECK(cudaMemcpyAsync(y.data(), c->psi.p, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(sq.data(), g.sqex, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(wj.data(), g.wjac, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(&mp, c->match_pt.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    // normalisation on the host here only to return u(r) for inspection; the SCF path normalises on the device
    double I = 0.;
    for (int i = 0; i < N; ++i) { y[i] *= sq[i]; I += wj[i] * y[i] * y[i]; }
    const double s_ = 1. / std::sqrt(I);
    for (int i = 0; i < N; ++i) u_out[i] = y[i] * s_;
    if (match_point) *match_point = mp;
    return 0;
}

int dftatom_poisson_solve(dftatom_ctx* c, int levels, double delta, double max_r, int n_dens, const int* Z, const double* rho,
                          double* U, int* vcycles_used)
{
    if (!c || !Z || !rho || !U || n_dens <= 0) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    DevBuf& dr = c->scratch[0]; DevBuf& dz = c->scratch[2]; DevBuf& dv = c->scratch[3];
    if ((rc = dr.ensure(sizeof(double) * (size_t)n_dens * N)) || (rc = dz.ensure(sizeof(double) * n_dens)) || (rc = dv.ensure(sizeof(int) * n_dens))) return rc;
    const std::vector<double> zbc(Z, Z + n_dens);            // the solvers take the boundary value as a double (an electron count)
    DFT_CHECK(cudaMemcpyAsync(dr.p, rho, sizeof(double) * (size_t)n_dens * N, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dz.p, zbc.data(), sizeof(double) * n_dens, cudaMemcpyHostToDevice, st));
    long long ld = N; bool streamed = false;
    if ((rc = poisson_cold(c, g, n_dens, dr.as<double>(), dz.as<double>(), dv.as<int>(), &ld, &streamed))) return rc;
    if (ld != N) DFT_CHECK(cudaMemcpy2DAsync(U, sizeof(double) * N, c->ubuf.p, sizeof(double) * ld, sizeof(double) * N, n_dens, cudaMemcpyDeviceToHost, st));
    else DFT_CHECK(cudaMemcpyAsync(U, c->ubuf.p, sizeof(double) * (size_t)n_dens * N, cudaMemcpyDeviceToHost, st));
    if (vcycles_used && streamed) for (int k = 0; k < n_dens; ++k) vcycles_used[k] = c->k.max_vcycles;
    else if (vcycles_used) DFT_CHECK(cudaMemcpyAsync(vcycles_used, dv.p, sizeof(int) * n_dens, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_poisson_increment(dftatom_ctx* c, int levels, double delta, double max_r, int n_dens, const double* rho, double* rho_prev,
                              double* U, const int* skip, int solver, int n_vcycles)
{
    if (!c || !rho || !rho_prev || !U || n_dens <= 0 || n_dens > 65535) { set_error("bad argument"); return DFTATOM_E_ARG; }
    if (levels < 8 || levels > 20) { set_error("levels must be in 8..20 (the SCF's range)"); return DFTATOM_E_BAD_OPTION; }
    if (solver < kIncDirect || solver > kIncColdForm) { set_error("solver must be 0 (direct), 1 (warm V-cycles) or 2 (increment form around the cold solvers)"); return DFTATOM_E_ARG; }
    if (solver != kIncDirect && (n_vcycles < 1 || n_vcycles > 1000)) { set_error("n_vcycles must be in 1..1000"); return DFTATOM_E_ARG; }
    if (c->k.poisson_exact || c->k.refine_vcycles || c->k.floor_stop) { set_error("the SCF solves no increment with poisson_exact, refine_vcycles or floor_stop set"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp; int rc = get_grid(c, levels, delta, max_r, &gp); if (rc) return rc;
    const GridDev g = *gp; const int N = g.N; cudaStream_t st = c->stream;
    const PoissonLevels lv = make_levels(levels);
    // the SCF's choices for a batch of n_dens atoms (solve_group)
    const bool stream = c->k.stream_poisson && n_dens >= c->k.stream_min_dens && levels >= c->k.stream_min_levels && levels > c->k.stream_mid_levels;
    const long long ldU = stream ? ((N + 3) & ~3) : N;
    if (solver == kIncDirect && g.coarse_direct == nullptr) { set_error("the direct solve needs 11..20 levels"); return DFTATOM_E_ARG; }
    if (solver == kIncWarmVcycles && (stream || !poisson_warm_supported(levels, delta) || g.coarse_tri == nullptr || (long long)lv.total < poisson_warm_scratch_doubles(levels))) {
        set_error("the warm V-cycle kernel needs 11..14 levels, delta > 0 and no stream-mode solver");
        return DFTATOM_E_ARG;
    }
    const StreamPlan splan = stream ? make_stream_plan(levels, n_dens, c->k.stream_mid_levels) : StreamPlan{};
    const size_t nN = (size_t)n_dens * N, nL = (size_t)n_dens * ldU;
    DevBuf& dr = c->scratch[0]; DevBuf& dp = c->scratch[1]; DevBuf& ds = c->scratch[2];
    if ((rc = dr.ensure(sizeof(double) * nN)) || (rc = dp.ensure(sizeof(double) * nN)) || (rc = ds.ensure(sizeof(int) * n_dens))
        || (rc = c->ubuf.ensure(sizeof(double) * nL)) || (rc = c->d_src.ensure(sizeof(double) * nL)) || (rc = c->d_u.ensure(sizeof(double) * nL))
        || (rc = c->phi.ensure(sizeof(double) * (size_t)n_dens * lv.total)) || (rc = c->src.ensure(sizeof(double) * (size_t)n_dens * lv.total))
        || (rc = c->team_bar.ensure(sizeof(unsigned) * (size_t)n_dens))) return rc;
    if (stream && (rc = c->stream_scratch.ensure(sizeof(double) * (size_t)splan.total))) return rc;
    DFT_CHECK(cudaMemcpyAsync(dr.p, rho, sizeof(double) * nN, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(dp.p, rho_prev, sizeof(double) * nN, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpy2DAsync(c->ubuf.p, sizeof(double) * ldU, U, sizeof(double) * N, sizeof(double) * N, n_dens, cudaMemcpyHostToDevice, st));
    if (skip) DFT_CHECK(cudaMemcpyAsync(ds.p, skip, sizeof(int) * n_dens, cudaMemcpyHostToDevice, st));
    // the arguments solve_group sets (the skip flags here: one int per density)
    PoissonArgs pa{};
    pa.n_dens = n_dens; pa.phi = c->phi.as<double>(); pa.src = c->src.as<double>(); pa.coarse_op = g.coarse_op;
    pa.skip = skip ? ds.as<int>() : nullptr; pa.skip_stride_bytes = (int)sizeof(int);
    pa.max_vcycles = c->k.max_vcycles; pa.u0 = c->u0.as<double>(); pa.n_sm = c->n_sm;
    pa.team_bar = c->k.team_poisson ? c->team_bar.as<unsigned>() : nullptr;
    WarmPoissonArgs ca{};
    ca.n_dens = n_dens; ca.rho = dr.as<double>(); ca.rho_stride = N; ca.rho_prev = dp.as<double>(); ca.U = c->ubuf.as<double>(); ca.ldU = ldU;
    ca.coarse_tri = g.coarse_tri; ca.skip = pa.skip; ca.skip_stride_bytes = pa.skip_stride_bytes;
    StreamSolveArgs sa{};
    sa.n_dens = n_dens; sa.rho_stride = N; sa.psrc = g.psrc; sa.ld0 = ldU; sa.scratch = c->stream_scratch.as<double>(); sa.coarse_op = g.coarse_op;
    sa.variant = c->k.stream_variant; sa.skip = pa.skip; sa.skip_stride_bytes = pa.skip_stride_bytes;
    long long nl = 0;
    poisson_increment(solver, g, lv, stream, splan, ca, pa, sa, c->d_src.as<double>(), c->d_u.as<double>(), n_vcycles, st, nl);
    DFT_CHECK(cudaMemcpy2DAsync(U, sizeof(double) * N, c->ubuf.p, sizeof(double) * ldU, sizeof(double) * N, n_dens, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(rho_prev, dp.p, sizeof(double) * nN, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

// The device part of dftatom_poisson_solve: the cold solve of n_dens densities d_rho [n_dens][N] with boundary values d_zbc [n_dens]
// (device arrays).  U = r V_H lands in c->ubuf with row stride *ld; d_vcycles [n_dens] receives the V-cycles run, except in stream mode
// (*streamed), which runs c->k.max_vcycles V-cycles for every density.
static int poisson_cold(dftatom_ctx* c, const GridDev& g, int n_dens, const double* d_rho, const double* d_zbc, int* d_vcycles, long long* ld_out,
                        bool* streamed)
{
    const int N = g.N, levels = g.L; const double delta = g.delta; cudaStream_t st = c->stream;
    const PoissonLevels lv = make_levels(levels);
    int rc;
    *ld_out = N; *streamed = false;
    if ((rc = c->phi.ensure(sizeof(double) * (size_t)n_dens * lv.total)) || (rc = c->src.ensure(sizeof(double) * (size_t)n_dens * lv.total))) return rc;
    PoissonArgs pa{};
    pa.n_dens = n_dens; pa.rho = d_rho; pa.Zbc = d_zbc; pa.phi = c->phi.as<double>(); pa.src = c->src.as<double>();
    pa.max_vcycles = c->k.max_vcycles; pa.floor_stop = c->k.floor_stop; pa.vcycles_used = d_vcycles;
    if ((rc = c->u0.ensure(sizeof(double) * (size_t)n_dens * N)) || (rc = c->ubuf.ensure(sizeof(double) * (size_t)n_dens * N))) return rc;
    pa.refine_vcycles = c->k.refine_vcycles; pa.u0 = c->u0.as<double>(); pa.u_out = c->ubuf.as<double>(); pa.coarse_op = g.coarse_op; pa.n_sm = c->n_sm;
    if ((rc = c->team_bar.ensure(sizeof(unsigned) * (size_t)n_dens))) return rc;
    pa.team_bar = c->k.team_poisson ? c->team_bar.as<unsigned>() : nullptr;
    if (c->k.profile) {
        if ((rc = c->scratch[5].ensure(sizeof(long long) * 128))) return rc;
        DFT_CHECK(cudaMemsetAsync(c->scratch[5].p, 0, sizeof(long long) * 128, st));
        pa.dbg = c->scratch[5].as<long long>();
    }
    if (n_dens > 65535) { set_error("at most 65535 densities per call"); return DFTATOM_E_ARG; }
    if (c->k.poisson_exact) {
        // bit-reproducible mode: the reference's FullCycle in its own operation order (poisson_exact.cu), 100 V-cycles
        if ((rc = c->exact_work.ensure(sizeof(double) * (size_t)n_dens * (size_t)exact_poisson_work_doubles(levels)))) return rc;
        ExactPoissonArgs xa{};
        xa.n_dens = n_dens; xa.L = levels; xa.delta = delta; xa.rho = d_rho; xa.rho_stride = N; xa.r = g.r; xa.pex = g.pex;
        xa.Zbc = d_zbc; xa.U = c->ubuf.as<double>(); xa.ldU = N; xa.work = c->exact_work.as<double>(); xa.max_vcycles = 100;
        xa.vcycles_used = d_vcycles;
        launch_poisson_exact(xa, st);
        return 0;
    }
    const bool stream = c->k.stream_poisson && n_dens >= c->k.stream_min_dens && levels >= c->k.stream_min_levels && levels > c->k.stream_mid_levels && levels <= 22 && c->k.refine_vcycles == 0 && !c->k.floor_stop && !c->k.profile;
    if (stream) {
        // grids beyond the chip: level visits streamed over all densities (poisson_stream.cu)
        const StreamPlan splan = make_stream_plan(levels, n_dens, c->k.stream_mid_levels);
        const long long ld = (N + 3) & ~3;
        if ((rc = c->stream_src0.ensure(sizeof(double) * (size_t)n_dens * ld)) || (rc = c->stream_scratch.ensure(sizeof(double) * (size_t)splan.total))) return rc;
        if ((rc = c->ubuf.ensure(sizeof(double) * (size_t)n_dens * ld))) return rc;
        StreamSolveArgs sa{};
        sa.n_dens = n_dens; sa.rho = d_rho; sa.rho_stride = N; sa.psrc = g.psrc; sa.src0 = c->stream_src0.as<double>();
        sa.U = c->ubuf.as<double>(); sa.ld0 = ld; sa.Zbc = d_zbc; sa.scratch = c->stream_scratch.as<double>(); sa.coarse_op = g.coarse_op;
        sa.n_v = c->k.max_vcycles; sa.warm = 0; sa.variant = c->k.stream_variant;
        launch_poisson_stream_solve(splan, delta, sa, st, nullptr);
        *ld_out = ld; *streamed = true;
        return 0;
    }
    launch_poisson_full(g, lv, pa, st);
    if (c->k.profile) {
        long long h[128];
        DFT_CHECK(cudaMemcpyAsync(h, pa.dbg, sizeof(h), cudaMemcpyDeviceToHost, st));
        DFT_CHECK(cudaStreamSynchronize(st));
        fprintf(stderr, "poisson cycles (CTA 0): setup %lld  solve %lld  +export %lld\n", h[98], h[96], h[97]);
        for (int l = 0; l < levels; ++l)
            fprintf(stderr, "  level %2d n=%7d  smooth %9lld (%lld visits)  restrict_to %8lld  prolong_from %8lld\n", l, (1 << (levels - l)), h[l], h[72 + l], h[24 + l], h[48 + l]);
        if (getenv("DFTATOM_DEBUG_WARM")) {      // the SCF's steady state: warm_vcycles V-cycles from the solution just computed
            DFT_CHECK(cudaMemsetAsync(pa.dbg, 0, sizeof(long long) * 128, st));
            pa.warm_vcycles = c->k.warm_vcycles;
            launch_poisson_full(g, lv, pa, st);
            DFT_CHECK(cudaMemcpyAsync(h, pa.dbg, sizeof(h), cudaMemcpyDeviceToHost, st));
            DFT_CHECK(cudaStreamSynchronize(st));
            fprintf(stderr, "warm start, %d V-cycles (CTA 0): setup %lld  solve %lld  +export %lld\n", c->k.warm_vcycles, h[98], h[96], h[97]);
            for (int l = 0; l < levels; ++l)
                fprintf(stderr, "  level %2d n=%7d  visits %9lld cycles (%lld visits)\n", l, (1 << (levels - l)), h[l], h[72 + l]);
        }
    }
    return 0;
}

long long dftatom_poisson_scratch_bytes(int levels, int n_dens)
{
    if (levels < 15 || levels > 22 || n_dens <= 0) return 0;
    long long t = 0;
    for (int mid = 11; mid <= 14; ++mid) t = std::max(t, make_stream_plan(levels, n_dens, mid).total);       // whatever "stream_mid_levels" is set to
    return (long long)sizeof(double) * t;
}

int dftatom_poisson_vcycles(dftatom_ctx* c, int levels, double delta, int n_dens, double* phi, const double* src, int n_cycles,
                            double* last_err)
{
    if (!c || !phi || !src || n_dens <= 0 || n_dens > 65535) return DFTATOM_E_ARG;
    if (levels < 1 || levels > 22 || !(delta >= 0.) || !std::isfinite(delta)) { set_error("bad grid: need 1 <= levels <= 22, finite delta >= 0"); return DFTATOM_E_BAD_OPTION; }
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const PoissonLevels lv = make_levels(levels);
    const int N = (1 << levels) + 1;
    int rc;
    if ((rc = c->phi.ensure(sizeof(double) * (size_t)n_dens * lv.total)) || (rc = c->src.ensure(sizeof(double) * (size_t)n_dens * lv.total))) return rc;
    DevBuf& de = c->scratch[3]; DevBuf& dp = c->scratch[0]; DevBuf& ds = c->scratch[1];
    if ((rc = de.ensure(sizeof(double) * n_dens))) return rc;
    if ((rc = dp.ensure(sizeof(double) * (size_t)n_dens * N)) || (rc = ds.ensure(sizeof(double) * (size_t)n_dens * N))) return rc;
    DFT_CHECK(cudaMemsetAsync(c->phi.p, 0, sizeof(double) * (size_t)n_dens * lv.total, st));
    DFT_CHECK(cudaMemsetAsync(c->src.p, 0, sizeof(double) * (size_t)n_dens * lv.total, st));
    DFT_CHECK(cudaMemcpyAsync(dp.p, phi, sizeof(double) * (size_t)n_dens * N, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemcpyAsync(ds.p, src, sizeof(double) * (size_t)n_dens * N, cudaMemcpyHostToDevice, st));
    launch_poisson_vcycles(lv, delta, n_dens, c->phi.as<double>(), c->src.as<double>(), dp.as<double>(), ds.as<double>(), n_cycles, de.as<double>(), st);
    DFT_CHECK(cudaMemcpyAsync(phi, dp.p, sizeof(double) * (size_t)n_dens * N, cudaMemcpyDeviceToHost, st));
    if (last_err) DFT_CHECK(cudaMemcpyAsync(last_err, de.p, sizeof(double) * n_dens, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_poisson_vcycles_dev(dftatom_ctx* c, int levels, double delta, int n_dens, void* d_phi, const void* d_src, long long ld,
                                void* d_scratch, long long scratch_bytes, int n_cycles, int fuse_tops, float* device_ms, long long* kernel_launches)
{
    if (!c || !d_phi || !d_src || !d_scratch || n_dens <= 0 || n_dens > 65535 || n_cycles <= 0) return DFTATOM_E_ARG;
    if (levels < 15 || levels > 22) { set_error("stream-mode V-cycles need 15 <= levels <= 22 (smaller grids are solved on chip: dftatom_poisson_vcycles)"); return DFTATOM_E_BAD_OPTION; }
    const long long N = (1ll << levels) + 1;
    if (ld < N || (ld & 1) || ((uintptr_t)d_phi & 15) || ((uintptr_t)d_src & 15) || ((uintptr_t)d_scratch & 15)) { set_error("ld must be even and >= N, pointers 16-byte aligned"); return DFTATOM_E_ARG; }
    const StreamPlan sp = make_stream_plan(levels, n_dens, c->k.stream_mid_levels);
    if (scratch_bytes < (long long)sizeof(double) * sp.total) { set_error("scratch too small"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    // dense operator of the coarse sub-cycle: depends on (levels, delta) only
    int rc;
    if ((rc = c->stream_G.ensure(sizeof(double) * 32 * 32))) return rc;
    if (c->stream_G_levels != levels || c->stream_G_delta != delta) {
        launch_coarse_op(levels, delta, c->stream_G.as<double>(), st);
        c->stream_G_levels = levels; c->stream_G_delta = delta;
    }
    cudaEvent_t e0, e1;
    DFT_CHECK(cudaEventCreate(&e0)); DFT_CHECK(cudaEventCreate(&e1));
    DFT_CHECK(cudaEventRecord(e0, st));
    long long nl = 0;
    launch_poisson_stream_vcycles(sp, delta, n_dens, (double*)d_phi, (const double*)d_src, ld, (double*)d_scratch, c->stream_G.as<double>(),
                                  n_cycles, fuse_tops, c->k.stream_variant, st, &nl);
    DFT_CHECK(cudaEventRecord(e1, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    float ms = 0.f;
    DFT_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (device_ms) *device_ms = ms;
    if (kernel_launches) *kernel_launches = nl;
    return 0;
}

int dftatom_vwn(dftatom_ctx* c, int n, const double* rho_a, const double* rho_b, double* va, double* vb, double* vexc, double* eexcdif)
{
    if (!c || !rho_a || !vexc || !eexcdif || n <= 0) return DFTATOM_E_ARG;
    if (rho_b && (!va || !vb)) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int rc;
    DevBuf& d = c->scratch[0];
    if ((rc = d.ensure(sizeof(double) * (size_t)n * 6))) return rc;
    double* p = d.as<double>();
    double* ra = p; double* rb = p + n; double* dva = p + 2 * (size_t)n; double* dvb = p + 3 * (size_t)n; double* dvx = p + 4 * (size_t)n; double* ded = p + 5 * (size_t)n;
    DFT_CHECK(cudaMemcpyAsync(ra, rho_a, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    if (rho_b) DFT_CHECK(cudaMemcpyAsync(rb, rho_b, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    launch_vwn(n, ra, rho_b ? rb : nullptr, dva, dvb, dvx, ded, st);
    if (rho_b) {
        DFT_CHECK(cudaMemcpyAsync(va, dva, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
        DFT_CHECK(cudaMemcpyAsync(vb, dvb, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    }
    DFT_CHECK(cudaMemcpyAsync(vexc, dvx, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(eexcdif, ded, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_simpson38(dftatom_ctx* c, double step, const double* v, int n, int n_rows, double* out)
{
    if (!c || !v || !out || n < 5 || n_rows <= 0) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int rc;
    DevBuf& d = c->scratch[0]; DevBuf& o = c->scratch[1];
    if ((rc = d.ensure(sizeof(double) * (size_t)n * n_rows)) || (rc = o.ensure(sizeof(double) * n_rows))) return rc;
    DFT_CHECK(cudaMemcpyAsync(d.p, v, sizeof(double) * (size_t)n * n_rows, cudaMemcpyHostToDevice, st));
    launch_simpson38(step, d.as<double>(), n, n_rows, o.as<double>(), st);
    DFT_CHECK(cudaMemcpyAsync(out, o.p, sizeof(double) * n_rows, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_xc_lda(dftatom_ctx* c, int functional, int n, const double* rho, double* vexc, double* eexcdif)
{
    if (!c || !rho || !vexc || !eexcdif || n <= 0 || functional < 0 || functional > 2) return DFTATOM_E_ARG;
    if (functional == 0) return dftatom_vwn(c, n, rho, nullptr, nullptr, nullptr, vexc, eexcdif);
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int rc;
    DevBuf& d = c->scratch[0];
    if ((rc = d.ensure(sizeof(double) * (size_t)n * 3))) return rc;
    double* p = d.as<double>();
    DFT_CHECK(cudaMemcpyAsync(p, rho, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    launch_chachiyo(n, p, functional == 2, p + n, p + 2 * (size_t)n, st);
    DFT_CHECK(cudaMemcpyAsync(vexc, p + n, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaMemcpyAsync(eexcdif, p + 2 * (size_t)n, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_integrate(dftatom_ctx* c, int rule, double step, const double* v, int n, int n_rows, double* out)
{
    if (!c || !v || !out || n_rows <= 0 || rule < 0 || rule > 4) return DFTATOM_E_ARG;
    // the size conditions the reference asserts (Integral.h:13, :27-28, :52-53, :77-78, :110)
    const bool ok = (rule == 0) ? n >= 2 : (rule == 1 || rule == 2) ? (n >= 5 && (n & 1)) : (rule == 3) ? (n > 4 && n % 4 == 1) : (n >= 3 && (n & 1) && n <= (1 << 22) + 1);
    if (!ok) { set_error("number of samples not admissible for this quadrature rule"); return DFTATOM_E_ARG; }
    DFT_CHECK(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int rc;
    DevBuf& d = c->scratch[0]; DevBuf& o = c->scratch[1];
    if ((rc = d.ensure(sizeof(double) * (size_t)n * n_rows)) || (rc = o.ensure(sizeof(double) * n_rows))) return rc;
    DFT_CHECK(cudaMemcpyAsync(d.p, v, sizeof(double) * (size_t)n * n_rows, cudaMemcpyHostToDevice, st));
    launch_integrate(rule, step, d.as<double>(), n, n_rows, o.as<double>(), st);
    DFT_CHECK(cudaMemcpyAsync(out, o.p, sizeof(double) * n_rows, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

int dftatom_radial_moments(dftatom_ctx* c, int levels, double delta, double max_r, const double* u, int n_rows, double* moments)
{
    if (!c || !u || !moments || n_rows <= 0) return DFTATOM_E_ARG;
    DFT_CHECK(cudaSetDevice(c->device));
    GridDev* gp = nullptr;
    int rc = get_grid(c, levels, delta, max_r, &gp);
    if (rc) return rc;
    const GridDev g = *gp;
    cudaStream_t st = c->stream;
    DevBuf& d = c->scratch[0]; DevBuf& o = c->scratch[1]; DevBuf& p = c->scratch[2]; DevBuf& t = c->scratch[3];
    if ((rc = d.ensure(sizeof(double) * (size_t)g.N * n_rows)) || (rc = o.ensure(sizeof(double) * DFTATOM_N_MOMENTS * (size_t)n_rows))
        || (rc = p.ensure(sizeof(double) * (size_t)radial_part_doubles(g.N, n_rows))) || (rc = t.ensure(sizeof(int) * (size_t)n_rows))) return rc;
    DFT_CHECK(cudaMemcpyAsync(d.p, u, sizeof(double) * (size_t)g.N * n_rows, cudaMemcpyHostToDevice, st));
    DFT_CHECK(cudaMemsetAsync(t.p, 0, sizeof(int) * (size_t)n_rows, st));
    launch_radial_orbitals(g, d.as<double>(), nullptr, 0, n_rows, nullptr, o.as<double>(), p.as<double>(), t.as<int>(), st);
    DFT_CHECK(cudaMemcpyAsync(moments, o.p, sizeof(double) * DFTATOM_N_MOMENTS * (size_t)n_rows, cudaMemcpyDeviceToHost, st));
    DFT_CHECK(cudaStreamSynchronize(st));
    DFT_CHECK(cudaGetLastError());
    return 0;
}

}  // extern "C"
