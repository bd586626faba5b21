// Radial Poisson multigrid, one CTA per density.
//
// Replaces (reference DFTAtom/) PoissonSolver.h:51-81 SolvePoissonNonUniform, :89-124 FullCycle, :155-159 VCycle and
// PoissonSolver.cpp:40-64 GaussSeidel, :66-77 IterateGaussSeidel, :80-106 Initialize, :110-123 Prolong, :126-157
// Restrict, :162-197 Ascend/Descend.
//
// The reference's smoother is a lexicographic in-place Gauss-Seidel sweep, i.e. the first-order recurrence
//     Phi_i <- a Phi_{i-1} + c_i ,   a = (1 + d_l/2)/2 ,   c_i = (S_i + (1 - d_l/2) Phi_{i+1}^old)/2 ,  d_l = δ 2^l .
// Every thread owns NPT consecutive nodes: it runs the recurrence locally with zero carry-in, the carries are
// resolved by a scan of the affine maps x -> a^NPT x + p (warp shuffles, then one shared-memory hop across warps),
// and the result is patched in.  That is the same sweep (same operator, same ordering), evaluated in O(NPT + log T)
// depth instead of O(N).  Because a ~ 1/2, a^k drops below FP64 resolution after ~64 nodes: the scans are truncated
// where the dropped terms are < 1e-19 relative.
//
// Where the time goes is latency, not flops (one solve = ~400 level visits of three dependent sweeps each), so:
//  * levels live in an owner-major layout (below): every access of a visit is unit-stride across the warp;
//  * a visit keeps the thread's nodes in registers for its three sweeps;
//  * levels with <= 512 nodes are run by warp 0 alone out of static shared memory: no block barrier;
//  * the sub-cycle below the 32-node level is one precomputed 32x32 operator (it depends on the grid only);
//  * Source_0 (read by every fine-grid sweep) and the mid levels sit in dynamic shared memory when they fit.
// The update norm of the reference's IterateGaussSeidel only drives its early exits; with a fixed number of sweeps it
// is evaluated once, for the last fine-grid sweep of the solve, and only when the caller asks for it.
#include "internal.h"
#include <algorithm>
#include <cmath>

namespace dft {

PoissonLevels make_levels(int L)
{
    PoissonLevels lv{};
    lv.L = L;
    int off = 0;
    for (int l = 0; l < L; ++l) {
        lv.size[l] = (1 << (L - l)) + 1;
        lv.off[l] = off;
        off += (lv.size[l] + 3) & ~3;      // keep every level 32-byte aligned
    }
    lv.total = off;
    return lv;
}

constexpr int kPT = 512;     // threads per CTA
constexpr int kLogPT = 9;
constexpr int kMaxNpt = 32;  // nodes per thread of a register-resident chunk (a chunk = T * npt consecutive nodes)
constexpr int kWarpLevelNodes = 512;    // levels up to this size are run by warp 0 alone (no block barrier)
constexpr int kWarpSmemDoubles = 2112;  // sum of the sizes of all levels with <= 512 owned nodes, 4-aligned each
constexpr double kTiny = 1e-19;   // carry terms below this (relative) are dropped from the truncated scans (FP64 eps = 1.1e-16)
constexpr int kMaxDynBytes = 180 * 1024;   // dynamic shared memory the solve kernels may ask for (static part: ~45 KB)

// ---------------------------------------------------------------------------------------------------------
// Owner-major level layout.  A level with n owned nodes (0..n-1; node n is the fixed right boundary) is run by T
// threads (T = 512: the CTA, or T = 32: warp 0 for the small levels).  It is cut into chunks of C = T * npt nodes,
// npt = clamp(n / T, 1, 32); inside a chunk thread t owns the npt consecutive nodes [t npt, (t+1) npt) and its k-th
// node is stored at  chunk_base + k T + t.  Every per-thread walk over "my nodes" is then a unit-stride access across
// the warp (coalesced in global memory, conflict-free in shared memory), and restriction / prolongation only touch
// the same thread's nodes plus one halo value.  Node n keeps slot n.
// ---------------------------------------------------------------------------------------------------------
struct Lay { int lgT, lg; };     // log2 T, log2 npt
__host__ __device__ inline Lay layout_of(int n)
{
    Lay y;
    y.lgT = (n <= kWarpLevelNodes) ? 5 : kLogPT;
    y.lg = 0;
    while (((1 << y.lgT) << (y.lg + 1)) <= n && y.lg < 5) ++y.lg;
    return y;
}
__host__ __device__ inline int slot(int i, Lay y)
{
    const int cm = ((1 << y.lgT) << y.lg) - 1;
    return (i & ~cm) | ((i & ((1 << y.lg) - 1)) << y.lgT) | ((i & cm) >> y.lg);
}
__host__ __device__ inline int unslot(int s, Lay y)
{
    const int cm = ((1 << y.lgT) << y.lg) - 1;
    const int j = s & cm;
    return (s & ~cm) | ((j & ((1 << y.lgT) - 1)) << y.lg) | (j >> y.lgT);
}

enum { kGlobal = 0, kDyn = 1, kWarp = 2 };     // where a level array lives

struct LevelConst {
    double d, a, bcoef;      // d_l = delta 2^l; a = (1 + d/2)/2; bcoef = (1 - d/2)/2       (PoissonSolver.cpp:56-57)
    double Ap[5];            // A^(2^j), A = a^npt: the multiplier of one thread's local affine map
    double B;                // A^32: the multiplier of one warp
    int nsteps;              // warp-scan steps that still matter (A^(2^j) >= kTiny)
    int n;                   // owned nodes
    Lay lay;
    int wp, ws;              // where Phi / Source live
    int op, os;              // their offsets (global: inside the density's hierarchy block; kDyn: in g_dyn; kWarp: in g_sm.w)
};

struct PoissonSmem {
    LevelConst lc[24];
    double* gphi; double* gsrc;   // this density's block of the global hierarchy arrays
    long long* dbg;      // optional cycle counters (development aid): [0,24) smooth, [24,48) restrict, [48,72) prolong, [72,96) visits
    int L, m, has_G;     // levels; level with 32 owned nodes that the dense operator starts from (valid when has_G)
    // team mode (large grids, few densities): team_G CTAs per density; rank 0 (the leader) runs the levels of <= 16384 nodes
    // as always, the others (workers) share every visit of the larger levels (big_visit); 0 / 1 = off
    int team_G, team_rank;
    unsigned* team_bar;  // arrival counter of this density's team (global memory, zero at launch)
    unsigned team_epoch;
    double wtot[16];     // per-warp totals of the local affine maps
    double edge[16];     // first node of every warp (old value for the left neighbour warp)
    double red[32];
    double carry;        // last new value of the previous chunk
    double apow[kMaxNpt]; // a^(k+1) of the level being visited (fused_block): the carry patch reads it instead of running its own product chain
    double bcast;
    unsigned long long updates;   // Gauss-Seidel node-updates performed by this CTA (work counter)
    double w[2 * kWarpSmemDoubles];   // the warp levels: Phi at [0, kWarpSmemDoubles), Source behind it
    double G[32 * 32];   // dense operator of the sub-cycle below the 32-node level, column-major G[j * 32 + i]
};

// File-scope shared variables: every access compiles to LDS/STS (a PoissonSmem& parameter would make them generic
// loads, which wait on the long scoreboard like global memory).
__shared__ PoissonSmem g_sm;
extern __shared__ double g_dyn[];

// one level array, wherever it lives
struct Ref {
    int w, off;
    double* g;
    static __device__ __forceinline__ Ref P(int l) { const LevelConst& c = g_sm.lc[l]; return Ref{ c.wp, c.op, g_sm.gphi }; }
    static __device__ __forceinline__ Ref S(int l) { const LevelConst& c = g_sm.lc[l]; return Ref{ c.ws, c.os, g_sm.gsrc }; }
    // global arrays are read with ld.cg: in team mode other CTAs write them between visits (L1 is not coherent across SMs)
    __device__ __forceinline__ double ld(int i) const { return w == kWarp ? g_sm.w[off + i] : (w == kDyn ? g_dyn[off + i] : __ldcg(g + off + i)); }
    __device__ __forceinline__ void st(int i, double v) const
    {
        if (w == kWarp) g_sm.w[off + i] = v; else if (w == kDyn) g_dyn[off + i] = v; else g[off + i] = v;
    }
};

__device__ __forceinline__ double block_sum(double v)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) g_sm.red[w] = v;
    __syncthreads();
    if (w == 0) {
        double t = (lane < (blockDim.x >> 5)) ? g_sm.red[lane] : 0.;
#pragma unroll
        for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) g_sm.bcast = t;
    }
    __syncthreads();
    return g_sm.bcast;
}

// ---------------------------------------------------------------------------------------------------------
// Register-resident visit of one chunk by the whole CTA: `sweeps` lexicographic Gauss-Seidel sweeps.
//   l, c0        : level and first slot of the chunk (Phi / Source: global memory or g_dyn, see LevelConst)
//   first        : the chunk starts with node 0 (fixed left boundary); otherwise left_new = new value of the node
//                  before the chunk
//   right_old    : value of the node after the chunk (old value: it is swept later, or it is the right boundary)
// ---------------------------------------------------------------------------------------------------------
template <int NPT, bool SRC_REGS>
__device__ __noinline__ void visit_regs(int l, int c0, int sweeps, bool first, double left_new, double right_old)
{
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const bool last_thr = (t == kPT - 1);
    const LevelConst& lc = g_sm.lc[l];
    const double a = lc.a, bcoef = lc.bcoef;
    const bool p_dyn = lc.wp == kDyn, s_dyn = lc.ws == kDyn;
    const int op = lc.op + c0, os = lc.os + c0;
    double* gp = g_sm.gphi + op;            // only dereferenced when the array is global
    const double* gs = g_sm.gsrc + os;
    double phi[NPT], src[SRC_REGS ? NPT : 1];
    if (p_dyn) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = g_dyn[op + k * kPT + t];
    } else {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = gp[k * kPT + t];
    }
    if (SRC_REGS) {
        if (s_dyn) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) src[k] = 0.5 * g_dyn[os + k * kPT + t];
        } else {
#pragma unroll
            for (int k = 0; k < NPT; ++k) src[k] = 0.5 * gs[k * kPT + t];
        }
    }
    // multipliers of the warp scan, pre-selected per lane (0 where the step does not apply or no longer matters)
    double Am[5];
    double Alane = 1.;                       // A^lane
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        Am[j] = (lane >= (1 << j) && j < lc.nsteps) ? lc.Ap[j] : 0.;
        if ((lane >> j) & 1) Alane *= lc.Ap[j];
    }
    const double B = lc.B;
    const int nsteps = lc.nsteps;
    if (t == 0) g_sm.updates += (unsigned long long)sweeps * (unsigned long long)(NPT * kPT);

    for (int sw = 0; sw < sweeps; ++sw) {
        // old value of the right neighbour's first node
        double nb = __shfl_down_sync(full, phi[0], 1);
        if (lane == 0) g_sm.edge[w] = phi[0];
        __syncthreads();
        if (lane == 31 && w + 1 < (kPT >> 5)) nb = g_sm.edge[w + 1];
        if (last_thr) nb = right_old;
        // local recurrence with zero carry-in, in place
        double x = 0.;
        if (SRC_REGS) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, src[k]);
                x = (first && t == 0 && k == 0) ? phi[0] : fma(a, x, c);      // node 0 keeps its boundary value
                phi[k] = x;
            }
        } else if (s_dyn) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, 0.5 * g_dyn[os + k * kPT + t]);
                x = (first && t == 0 && k == 0) ? phi[0] : fma(a, x, c);
                phi[k] = x;
            }
        } else {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, 0.5 * gs[k * kPT + t]);
                x = (first && t == 0 && k == 0) ? phi[0] : fma(a, x, c);
                phi[k] = x;
            }
        }
        // warp scan of the totals (uniform multiplier): P_lane = sum_j A^(lane-j) p_j
        double P = x;
        P = fma(Am[0], __shfl_up_sync(full, P, 1), P);
        if (nsteps > 1) {
            P = fma(Am[1], __shfl_up_sync(full, P, 2), P);
            if (nsteps > 2) {
                P = fma(Am[2], __shfl_up_sync(full, P, 4), P);
                P = fma(Am[3], __shfl_up_sync(full, P, 8), P);
                P = fma(Am[4], __shfl_up_sync(full, P, 16), P);
            }
        }
        if (lane == 31) g_sm.wtot[w] = P;
        __syncthreads();
        // carry into this warp: sum_k B^(k-1) W_(w-k)  (+ B^w left_new), truncated
        double carry = 0.;
        {
            double bp = 1.;
            int k = 1;
            for (; k <= w && bp >= kTiny; ++k) { carry = fma(bp, g_sm.wtot[w - k], carry); bp *= B; }
            if (k > w && bp >= kTiny && !first) carry = fma(bp, left_new, carry);
        }
        double Pex = __shfl_up_sync(full, P, 1);
        if (lane == 0) Pex = 0.;
        double cin = fma(Alane, carry, Pex);                   // new value of the node before this thread's first node
        if (first && t == 0) cin = 0.;
        double q = a;
#pragma unroll
        for (int k = 0; k < NPT; ++k) { phi[k] = fma(q, cin, phi[k]); q *= a; }
    }
    if (p_dyn) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) g_dyn[op + k * kPT + t] = phi[k];
    } else {
#pragma unroll
        for (int k = 0; k < NPT; ++k) gp[k * kPT + t] = phi[k];
    }
    if (last_thr) g_sm.carry = phi[NPT - 1];
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------
// The same visit for a level of <= 1024 owned nodes, executed by warp 0 alone (no block barrier): lane owns NPT
// consecutive nodes (owner-major layout with T = 32, static shared memory).  n < 32: one node per lane, n lanes active.
// ---------------------------------------------------------------------------------------------------------
template <int NPT, bool SRC_REGS>
__device__ __noinline__ void visit_warp(int l, int sweeps)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const LevelConst& lc = g_sm.lc[l];
    const int n = lc.n, op = lc.op, os = lc.os;
    const bool active = lane * NPT < n;
    const bool last_lane = ((lane + 1) * NPT >= n) && active;
    const double a = lc.a, bcoef = lc.bcoef;
    const double right_bc = g_sm.w[op + n];
    double phi[NPT], src[SRC_REGS ? NPT : 1];
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
        phi[k] = active ? g_sm.w[op + k * 32 + lane] : 0.;
        if (SRC_REGS) src[k] = active ? 0.5 * g_sm.w[os + k * 32 + lane] : 0.;
    }
    double Am[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) Am[j] = (lane >= (1 << j) && j < lc.nsteps) ? lc.Ap[j] : 0.;
    const int nsteps = lc.nsteps;
    for (int sw = 0; sw < sweeps; ++sw) {
        double nb = __shfl_down_sync(full, phi[0], 1);
        if (last_lane) nb = right_bc;
        double x = 0.;
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, SRC_REGS ? src[k] : 0.5 * g_sm.w[os + k * 32 + lane]);
            x = (lane == 0 && k == 0) ? phi[0] : fma(a, x, c);
            phi[k] = x;
        }
        double P = active ? x : 0.;
        P = fma(Am[0], __shfl_up_sync(full, P, 1), P);
        if (nsteps > 1) {
            P = fma(Am[1], __shfl_up_sync(full, P, 2), P);
            if (nsteps > 2) {
                P = fma(Am[2], __shfl_up_sync(full, P, 4), P);
                P = fma(Am[3], __shfl_up_sync(full, P, 8), P);
                P = fma(Am[4], __shfl_up_sync(full, P, 16), P);
            }
        }
        double cin = __shfl_up_sync(full, P, 1);
        if (lane == 0) cin = 0.;
        double q = a;
#pragma unroll
        for (int k = 0; k < NPT; ++k) { phi[k] = fma(q, cin, phi[k]); q *= a; }
    }
    if (active) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) g_sm.w[op + k * 32 + lane] = phi[k];
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
// Fused visits.  Restriction and prolongation only need the thread's own nodes plus one halo value (owner-major layout,
// coarse node i <-> fine node 2i belong to the same thread), so they are folded into the visit that has the level in
// registers anyway:
//   kLoadPhi     : Phi_l starts from memory (otherwise from zero: a level entered by restriction)
//   kProlongIn   : Phi_l += P Phi_{l+1} before sweeping                      (Prolong, PoissonSolver.cpp:110-123)
//   kRestrictOut : after sweeping, Source_{l+1} = 4 R (residual) (- d_{l+1} first-difference term); Phi_{l+1} is implicitly
//                  zero: the visit of level l+1 that follows starts from zero   (Restrict, PoissonSolver.cpp:126-157)
// A V-cycle is then one visit per level and leg, and a level costs one load and one store of Phi per visit instead of
// the separate smoothing / restriction / prolongation passes.  An up-visit followed by the down-visit of the next cycle
// on the same level is ONE visit with 6 sweeps (kLoadPhi | kProlongIn | kRestrictOut).
// ---------------------------------------------------------------------------------------------------------
enum { kLoadPhi = 1, kProlongIn = 2, kRestrictOut = 4 };

template <int NPT, bool SRC_REGS>
__device__ __noinline__ void fused_block(int l, int flags, int sweeps)
{
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    constexpr int NC = NPT / 2;
    const bool last_thr = (t == kPT - 1);
    const LevelConst& lc = g_sm.lc[l];
    const LevelConst& lcc = g_sm.lc[l + 1];
    const double a = lc.a, bcoef = lc.bcoef;
    const int n = NPT * kPT;
    const Ref P = Ref::P(l), S = Ref::S(l);
    double phi[NPT], src[SRC_REGS ? NPT : 1];
    double right = 0.;
    if (flags & kLoadPhi) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = P.ld(k * kPT + t);
        right = P.ld(n);
    } else {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = 0.;
    }
    if (flags & kProlongIn) {
        const Ref Pc = Ref::P(l + 1);
        const Lay yc = lcc.lay;
        double corr[NC + 1];
#pragma unroll
        for (int m = 0; m <= NC; ++m) corr[m] = Pc.ld(slot(t * NC + m, yc));      // m = NC: the right neighbour's first node (or the boundary)
#pragma unroll
        for (int m = 0; m < NC; ++m) {
            phi[2 * m] += corr[m];
            phi[2 * m + 1] += 0.5 * (corr[m] + corr[m + 1]);
        }
        right += Pc.ld(lcc.n);
    }
    if (SRC_REGS) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) src[k] = 0.5 * S.ld(k * kPT + t);
    }
    const bool s_dyn = lc.ws == kDyn;
    const int os = lc.os;
    const double* gs = g_sm.gsrc + os;
    double Am[5];
    double Alane = 1.;                       // A^lane
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        Am[j] = (lane >= (1 << j) && j < lc.nsteps) ? lc.Ap[j] : 0.;
        if ((lane >> j) & 1) Alane *= lc.Ap[j];
    }
    const double B = lc.B;
    const int nsteps = lc.nsteps;
    if (t == 0) g_sm.updates += (unsigned long long)sweeps * (unsigned long long)(n - 1);
    if (t < NPT) { double q = a; for (int j = 0; j < t; ++j) q *= a; g_sm.apow[t] = q; }      // same products, same order, as a running q *= a
    double cin = 0.;
    for (int sw = 0; sw < sweeps; ++sw) {
        double nb = __shfl_down_sync(full, phi[0], 1);
        if (lane == 0) g_sm.edge[w] = phi[0];
        __syncthreads();
        if (lane == 31 && w + 1 < (kPT >> 5)) nb = g_sm.edge[w + 1];
        if (last_thr) nb = right;
        double x = 0.;
        if (SRC_REGS) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, src[k]);
                x = (t == 0 && k == 0) ? phi[0] : fma(a, x, c);      // node 0 keeps its boundary value
                phi[k] = x;
            }
        } else if (s_dyn) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, 0.5 * g_dyn[os + k * kPT + t]);
                x = (t == 0 && k == 0) ? phi[0] : fma(a, x, c);
                phi[k] = x;
            }
        } else {
#pragma unroll
            for (int k = 0; k < NPT; ++k) {
                const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, 0.5 * __ldcg(gs + k * kPT + t));
                x = (t == 0 && k == 0) ? phi[0] : fma(a, x, c);
                phi[k] = x;
            }
        }
        double Pw = x;
        Pw = fma(Am[0], __shfl_up_sync(full, Pw, 1), Pw);
        if (nsteps > 1) {
            Pw = fma(Am[1], __shfl_up_sync(full, Pw, 2), Pw);
            if (nsteps > 2) {
                Pw = fma(Am[2], __shfl_up_sync(full, Pw, 4), Pw);
                Pw = fma(Am[3], __shfl_up_sync(full, Pw, 8), Pw);
                Pw = fma(Am[4], __shfl_up_sync(full, Pw, 16), Pw);
            }
        }
        if (lane == 31) g_sm.wtot[w] = Pw;
        __syncthreads();
        // carry into this warp: the new value of the previous warp's last node; terms from further back carry B = A^32 per warp,
        // below FP64 resolution for every block level (a^64 < 1e-19), so the general loop almost never runs
        double carry = (w > 0) ? g_sm.wtot[w - 1] : 0.;
        if (B >= kTiny) {
            double bp = B;
            for (int k = 2; k <= w && bp >= kTiny; ++k) { carry = fma(bp, g_sm.wtot[w - k], carry); bp *= B; }
        }
        double Pex = __shfl_up_sync(full, Pw, 1);
        if (lane == 0) Pex = 0.;
        cin = fma(Alane, carry, Pex);                           // new value of the node before this thread's first node
        if (t == 0) cin = 0.;
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = fma(g_sm.apow[k], cin, phi[k]);
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) P.st(k * kPT + t, phi[k]);
    if (t == 0) P.st(n, right);
    if (flags & kRestrictOut) {
        const Ref Sc = Ref::S(l + 1);
        const Lay yc = lcc.lay;
        const double dc = lcc.d;
#pragma unroll
        for (int m = 0; m < NC; ++m) {
            const int k = 2 * m;
            const double lft = (m == 0) ? cin : phi[k - 1], mid = phi[k], rgt = phi[k + 1];
            const double sv = SRC_REGS ? 2. * src[k] : S.ld(k * kPT + t);
            double v = 4. * (sv + lft - 2. * mid + rgt) - dc * (rgt - lft);
            if (t == 0 && m == 0) v = 0.;
            Sc.st(slot(t * NC + m, yc), v);
        }
        if (t == 0) Sc.st(lcc.n, 0.);
    }
    __syncthreads();
}

// the same for the levels run by warp 0 (T = 32, static shared memory, 64 <= n <= 512, NPT = n / 32)
template <int NPT, bool SRC_REGS>
__device__ __noinline__ void fused_warp(int l, int flags, int sweeps)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    constexpr int NC = NPT / 2;
    const LevelConst& lc = g_sm.lc[l];
    const LevelConst& lcc = g_sm.lc[l + 1];
    const int n = NPT * 32, op = lc.op, os = lc.os, opc = lcc.op, osc = lcc.os;
    const double a = lc.a, bcoef = lc.bcoef;
    double phi[NPT], src[SRC_REGS ? NPT : 1];
    double right = 0.;
    if (flags & kLoadPhi) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = g_sm.w[op + k * 32 + lane];
        right = g_sm.w[op + n];
    } else {
#pragma unroll
        for (int k = 0; k < NPT; ++k) phi[k] = 0.;
    }
    if (flags & kProlongIn) {
        // coarse level: NC nodes per lane (NC >= 1), owner-major with T = 32: node lane NC + m at slot m 32 + lane
        double corr[NC + 1];
#pragma unroll
        for (int m = 0; m < NC; ++m) corr[m] = g_sm.w[opc + m * 32 + lane];
        corr[NC] = (lane == 31) ? g_sm.w[opc + lcc.n] : g_sm.w[opc + lane + 1];      // first node of the right neighbour / boundary
#pragma unroll
        for (int m = 0; m < NC; ++m) {
            phi[2 * m] += corr[m];
            phi[2 * m + 1] += 0.5 * (corr[m] + corr[m + 1]);
        }
        right += g_sm.w[opc + lcc.n];
    }
    if (SRC_REGS) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) src[k] = 0.5 * g_sm.w[os + k * 32 + lane];
    }
    double Am[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) Am[j] = (lane >= (1 << j) && j < lc.nsteps) ? lc.Ap[j] : 0.;
    const int nsteps = lc.nsteps;
    if (lane == 0) g_sm.updates += (unsigned long long)sweeps * (unsigned long long)(n - 1);
    double cin = 0.;
    for (int sw = 0; sw < sweeps; ++sw) {
        double nb = __shfl_down_sync(full, phi[0], 1);
        if (lane == 31) nb = right;
        double x = 0.;
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, SRC_REGS ? src[k] : 0.5 * g_sm.w[os + k * 32 + lane]);
            x = (lane == 0 && k == 0) ? phi[0] : fma(a, x, c);
            phi[k] = x;
        }
        double Pw = x;
        Pw = fma(Am[0], __shfl_up_sync(full, Pw, 1), Pw);
        if (nsteps > 1) {
            Pw = fma(Am[1], __shfl_up_sync(full, Pw, 2), Pw);
            if (nsteps > 2) {
                Pw = fma(Am[2], __shfl_up_sync(full, Pw, 4), Pw);
                Pw = fma(Am[3], __shfl_up_sync(full, Pw, 8), Pw);
                Pw = fma(Am[4], __shfl_up_sync(full, Pw, 16), Pw);
            }
        }
        cin = __shfl_up_sync(full, Pw, 1);
        if (lane == 0) cin = 0.;
        double q = a;
#pragma unroll
        for (int k = 0; k < NPT; ++k) { phi[k] = fma(q, cin, phi[k]); q *= a; }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) g_sm.w[op + k * 32 + lane] = phi[k];
    if (lane == 0) g_sm.w[op + n] = right;
    if (flags & kRestrictOut) {
        const double dc = lcc.d;
#pragma unroll
        for (int m = 0; m < NC; ++m) {
            const int k = 2 * m;
            const double lft = (m == 0) ? cin : phi[k - 1], mid = phi[k], rgt = phi[k + 1];
            const double sv = SRC_REGS ? 2. * src[k] : g_sm.w[os + k * 32 + lane];
            double v = 4. * (sv + lft - 2. * mid + rgt) - dc * (rgt - lft);
            if (lane == 0 && m == 0) v = 0.;
            g_sm.w[osc + m * 32 + lane] = v;
        }
        if (lane == 0) g_sm.w[osc + lcc.n] = 0.;
    }
    __syncwarp();
}

// Restrict, PoissonSolver.cpp:126-157: coarse slots are walked in storage order (coalesced); the three fine nodes of a
// coarse node belong to the same thread's chunk (plus one halo node of the left neighbour)
__device__ __forceinline__ void restrict_nodes(Ref pf, Ref sf, Lay yf, Ref pc, Ref sc, Lay yc, int nc, double dc, int tid, int nthr)
{
    for (int s = tid; s < nc; s += nthr) {          // nc = size of the coarse level; slot nc-1 is its right boundary
        const int i = unslot(s, yc);
        double v = 0.;
        if (i > 0 && i < nc - 1) {
            const int k = 2 * i;
            const double lft = pf.ld(slot(k - 1, yf)), mid = pf.ld(slot(k, yf)), rgt = pf.ld(slot(k + 1, yf));
            v = 4. * (sf.ld(slot(k, yf)) + lft - 2. * mid + rgt) - dc * (rgt - lft);
        }
        pc.st(s, 0.);
        sc.st(s, v);
    }
}

__device__ __forceinline__ void prolong_nodes(Ref pc, Lay yc, Ref pf, Lay yf, int nc, int tid, int nthr)
{   // Prolong, PoissonSolver.cpp:110-123
    for (int s = tid; s < nc; s += nthr) {
        const int i = unslot(s, yc);
        const double c = pc.ld(s);
        const int s2 = slot(2 * i, yf);
        pf.st(s2, pf.ld(s2) + c);
        if (i > 0) {
            const int s1 = slot(2 * i - 1, yf);
            pf.st(s1, pf.ld(s1) + 0.5 * (pc.ld(slot(i - 1, yc)) + c));
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// One multigrid hierarchy of one density.  All state is in g_sm; the functions below are called by all threads of the
// CTA.  The heavy bodies are __noinline__ functions of the level index only (a fat inlined dispatcher costs hundreds of
// spill instructions per call), the wrappers that carry the per-thread `pending` flag are inlined.
// ---------------------------------------------------------------------------------------------------------
struct Ctl {
    bool pending;        // warp 0 wrote coarse levels that the other warps have not synchronised with yet
    bool small_done;     // team mode: the leader has worked on its own levels since the last team barrier
};

__device__ __forceinline__ void block_begin(Ctl& ctl) { if (ctl.pending) { __syncthreads(); ctl.pending = false; } }

// per-level constants and placement (threads 0..L-1 fill one level each; every thread computes the same placement)
constexpr int kTeamLevelNodes = kPT * kMaxNpt;     // team mode: levels with more nodes than this are shared by the team

__device__ __noinline__ void hierarchy_setup(const PoissonLevels& lv, double delta, double* gphi, double* gsrc, int dyn_doubles,
                                             const double* Gg, long long* dbg, int team_G = 1, int team_rank = 0, unsigned* team_bar = nullptr)
{
    const int l = threadIdx.x;
    if (l < lv.L) {
        LevelConst c;
        c.n = lv.size[l] - 1;
        c.d = delta * (double)(1 << l);
        c.a = 0.5 * (1. + 0.5 * c.d);
        c.bcoef = 0.5 * (1. - 0.5 * c.d);
        c.lay = layout_of(c.n);
        double A = c.a;
        for (int k = 0; k < c.lay.lg; ++k) A *= A;
        c.Ap[0] = A;
        for (int j = 1; j < 5; ++j) c.Ap[j] = c.Ap[j - 1] * c.Ap[j - 1];
        c.B = c.Ap[4] * c.Ap[4];
        c.nsteps = 5;
        for (int j = 4; j >= 0; --j) if (c.Ap[j] < kTiny) c.nsteps = j;
        c.wp = c.ws = kGlobal; c.op = c.os = lv.off[l];
        // warp levels: static shared memory
        int woff = 0;
        for (int k = 0; k < lv.L; ++k) {
            const int nk = lv.size[k] - 1;
            if (nk > kWarpLevelNodes) continue;
            if (k == l) { c.wp = c.ws = kWarp; c.op = woff; c.os = kWarpSmemDoubles + woff; }
            woff += (nk + 4) & ~3;
        }
        // dynamic shared memory: Source_0 first (every fine-grid sweep streams it), then whole levels, coarsest first
        int avail = dyn_doubles, doff = 0;
        const int n0 = lv.size[0] - 1;
        bool src0_dyn = false;
        if (n0 > kWarpLevelNodes && ((n0 + 4) & ~3) <= avail) {
            src0_dyn = true;
            if (l == 0) { c.ws = kDyn; c.os = doff; }
            doff += (n0 + 4) & ~3; avail -= (n0 + 4) & ~3;
        }
        for (int k = lv.L - 1; k >= 0; --k) {
            const int nk = lv.size[k] - 1;
            if (nk <= kWarpLevelNodes) continue;
            const int one = (nk + 4) & ~3;
            const int need = (k == 0 && src0_dyn) ? one : 2 * one;
            if (need > avail) break;
            if (k == l) {
                c.wp = kDyn; c.op = doff;
                if (!(k == 0 && src0_dyn)) { c.ws = kDyn; c.os = doff + one; }
            }
            doff += need; avail -= need;
        }
        if (team_G > 1) {
            // the team's levels: natural node order in global memory (every CTA reads and writes contiguous windows);
            // the first level below them is written by the workers and read by the leader: global memory as well
            if (c.n > kTeamLevelNodes) { c.lay.lgT = 0; c.lay.lg = 0; c.wp = c.ws = kGlobal; c.op = c.os = lv.off[l]; }
            else if (l > 0 && lv.size[l - 1] - 1 > kTeamLevelNodes) { c.wp = c.ws = kGlobal; c.op = c.os = lv.off[l]; }
        }
        g_sm.lc[l] = c;
    }
    if (threadIdx.x == 0) {
        g_sm.gphi = gphi; g_sm.gsrc = gsrc; g_sm.dbg = dbg;
        g_sm.L = lv.L; g_sm.m = lv.L - 5; g_sm.has_G = (Gg != nullptr && lv.L - 5 >= 1) ? 1 : 0;
        g_sm.updates = 0;
        g_sm.team_G = team_G; g_sm.team_rank = team_rank; g_sm.team_bar = team_bar; g_sm.team_epoch = 0;
    }
    if (Gg != nullptr && lv.L - 5 >= 1) for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) g_sm.G[i] = Gg[i];
    __syncthreads();
}

// IterateGaussSeidel(l, ., sweeps) without the early exit, levels run by warp 0
__device__ __noinline__ void smooth_warp(int l, int sweeps)
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    const LevelConst& c = g_sm.lc[l];
    if (threadIdx.x == 0) g_sm.updates += (unsigned long long)sweeps * (unsigned long long)(c.n - 1);
    switch (c.lay.lg) {
        case 4: visit_warp<16, true>(l, sweeps); break;
        case 3: visit_warp<8, true>(l, sweeps); break;
        case 2: visit_warp<4, true>(l, sweeps); break;
        case 1: visit_warp<2, true>(l, sweeps); break;
        default: visit_warp<1, true>(l, sweeps); break;
    }
    if (g_sm.dbg && threadIdx.x == 0) { g_sm.dbg[l] += clock64() - t0; g_sm.dbg[72 + l] += 1; }
}
// ... levels run by the whole CTA
__device__ __noinline__ void smooth_block(int l, int sweeps)
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    const LevelConst& c = g_sm.lc[l];
    const int n = c.n;
    const Ref pr = Ref::P(l);
    if (n > kPT * kMaxNpt) {
        // multi-chunk level: one sweep at a time, chunk after chunk (carry = new value of the previous chunk's last node)
        const int C = kPT * kMaxNpt;
        for (int k = 0; k < sweeps; ++k) {
            double left = 0.;
            for (int c0 = 0; c0 < n; c0 += C) {
                const double right = pr.ld(c0 + C);      // first node of the next chunk (slot c0 + C) or the boundary node n
                visit_regs<32, false>(l, c0, 1, c0 == 0, left, right);
                left = g_sm.carry;
            }
        }
    } else {
        const double right = pr.ld(n);
        switch (c.lay.lg) {
            case 5: visit_regs<32, false>(l, 0, sweeps, true, 0., right); break;
            case 4: visit_regs<16, true>(l, 0, sweeps, true, 0., right); break;
            case 3: visit_regs<8, true>(l, 0, sweeps, true, 0., right); break;
            case 2: visit_regs<4, true>(l, 0, sweeps, true, 0., right); break;
            default: visit_regs<2, true>(l, 0, sweeps, true, 0., right); break;   // n = 1024 (n <= 512 are warp levels)
        }
    }
    if (g_sm.dbg && threadIdx.x == 0) { g_sm.dbg[l] += clock64() - t0; g_sm.dbg[72 + l] += 1; }
}
__device__ __forceinline__ void smooth(Ctl& ctl, int l, int sweeps)
{
    if (g_sm.lc[l].wp == kWarp) {
        if (threadIdx.x < 32) smooth_warp(l, sweeps);
        ctl.pending = true;
    } else {
        block_begin(ctl);
        smooth_block(l, sweeps);
    }
}

__device__ __noinline__ void restrict_impl(int l, int tid, int nthr)       // level l-1 -> l
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    const LevelConst& cf = g_sm.lc[l - 1];
    const LevelConst& cc = g_sm.lc[l];
    restrict_nodes(Ref::P(l - 1), Ref::S(l - 1), cf.lay, Ref::P(l), Ref::S(l), cc.lay, cc.n + 1, cc.d, tid, nthr);
    if (nthr == 32) __syncwarp(); else __syncthreads();
    if (g_sm.dbg && threadIdx.x == 0) g_sm.dbg[24 + l] += clock64() - t0;
}
__device__ __forceinline__ void restrict_to(Ctl& ctl, int l)
{
    if (g_sm.lc[l - 1].wp == kWarp) {                           // both levels belong to warp 0
        if (threadIdx.x < 32) restrict_impl(l, threadIdx.x, 32);
        ctl.pending = true;
    } else {
        block_begin(ctl);
        restrict_impl(l, threadIdx.x, kPT);
    }
}
__device__ __noinline__ void prolong_impl(int l, int tid, int nthr)        // level l -> l-1
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    const LevelConst& cf = g_sm.lc[l - 1];
    const LevelConst& cc = g_sm.lc[l];
    prolong_nodes(Ref::P(l), cc.lay, Ref::P(l - 1), cf.lay, cc.n + 1, tid, nthr);
    if (nthr == 32) __syncwarp(); else __syncthreads();
    if (g_sm.dbg && threadIdx.x == 0) g_sm.dbg[48 + l] += clock64() - t0;
}
__device__ __forceinline__ void prolong_from(Ctl& ctl, int l)
{
    if (g_sm.lc[l - 1].wp == kWarp) {
        if (threadIdx.x < 32) prolong_impl(l, threadIdx.x, 32);
        ctl.pending = true;
    } else {
        block_begin(ctl);
        prolong_impl(l, threadIdx.x, kPT);
    }
}
// phi_m = G src_m : the whole sub-cycle  smooth(m) restrict ... smooth(c) ... prolong smooth(m)  entered with phi_m = 0
// is a fixed linear map of the 31 interior source values (it depends on the grid only; built by coarse_op_kernel)
__device__ __noinline__ void dense_apply_warp()
{
    const LevelConst& c = g_sm.lc[g_sm.m];
    const int i = threadIdx.x;
    double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        a0 = fma(g_sm.G[(j + 0) * 32 + i], g_sm.w[c.os + j + 0], a0);
        a1 = fma(g_sm.G[(j + 1) * 32 + i], g_sm.w[c.os + j + 1], a1);
        a2 = fma(g_sm.G[(j + 2) * 32 + i], g_sm.w[c.os + j + 2], a2);
        a3 = fma(g_sm.G[(j + 3) * 32 + i], g_sm.w[c.os + j + 3], a3);
    }
    g_sm.w[c.op + i] = (a0 + a1) + (a2 + a3);      // row 0 of G is zero: the left boundary stays 0
    if (i == 0) g_sm.w[c.op + 32] = 0.;            // a level entered by restriction has zero boundaries
    __syncwarp();
}
__device__ __forceinline__ void to_coarse(Ctl& ctl, int from, int to)      // "Ascend", PoissonSolver.cpp:162-171
{
    for (int l = from; l < to; ++l) { smooth(ctl, l, 3); restrict_to(ctl, l + 1); }
    smooth(ctl, to, 3);
}
__device__ __forceinline__ void to_fine(Ctl& ctl, int from, int to)        // "Descend", PoissonSolver.cpp:173-186
{
    for (int l = from; l > to; --l) { prolong_from(ctl, l); smooth(ctl, l - 1, 3); }
}
// to_coarse(from, c) followed by to_fine(c, to).  With norm_scratch (N doubles of global memory) and to == 0 it also
// returns sqrt(sum (old - new)^2) of the last fine-grid sweep (the reference's IterateGaussSeidel norm).
__device__ __noinline__ double cycle(Ctl& ctl, int from, int to, double* norm_scratch)
{
    const int c = g_sm.L - 1, m = g_sm.m;
    int top;
    if (g_sm.has_G && from < m && to < m) {
        for (int l = from; l < m; ++l) { smooth(ctl, l, 3); restrict_to(ctl, l + 1); }
        if (threadIdx.x < 32) dense_apply_warp();
        ctl.pending = true;
        top = m;
    } else {
        to_coarse(ctl, from, c);
        top = c;
    }
    const bool norm = norm_scratch != nullptr && to == 0 && top > 0;
    for (int l = top; l > to; --l) {
        prolong_from(ctl, l);
        if (norm && l == 1) break;
        smooth(ctl, l - 1, 3);
    }
    if (!norm) return 0.;
    smooth(ctl, 0, 2);
    block_begin(ctl);
    const Ref p0 = Ref::P(0);
    const int N = g_sm.lc[0].n + 1;
    for (int s = threadIdx.x; s < N; s += blockDim.x) norm_scratch[s] = p0.ld(s);
    __syncthreads();
    smooth(ctl, 0, 1);
    block_begin(ctl);
    double e2 = 0.;
    for (int s = threadIdx.x; s < N; s += blockDim.x) { const double dif = norm_scratch[s] - p0.ld(s); e2 = fma(dif, dif, e2); }
    return sqrt(block_sum(e2));
}
// ---------------------------------------------------------------------------------------------------------
// Team mode.  A level visit (3 or 6 lexicographic sweeps) only needs old values up to `sweeps` nodes to the right of a
// node and, because a ~ 1/2, new values up to ~64 nodes to its left per sweep (a^64 < 1e-19).  A slab of a large level
// can therefore be swept by one CTA on its own, from a window that extends the slab by a halo (HL = 128 / 256 nodes on
// the left for 3 / 6 sweeps, 8 on the right) whose ends are held fixed at their old values: inside the slab the result is
// the lexicographic sweep of the whole level to FP64 resolution, and the CTAs of a team need no carry exchange inside a
// visit - only a barrier between visits.  The window lives in shared memory (coalesced global reads and writes).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool team_level(int l) { return g_sm.team_G > 1 && g_sm.lc[l].n > kTeamLevelNodes; }

__device__ __forceinline__ void team_barrier()
{
    if (g_sm.team_G <= 1) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned target = (unsigned)g_sm.team_G * (++g_sm.team_epoch);
        atomicAdd(g_sm.team_bar, 1u);
        while (*(volatile unsigned*)g_sm.team_bar < target) { }
        __threadfence();
    }
    __syncthreads();
}

constexpr int kHaloR = 8;
__host__ __device__ inline int team_halo_left(int sweeps) { return sweeps > 3 ? 256 : 128; }
// nodes per thread of the window of a team visit: the smallest of 4, 8, 16 whose slabs cover the level with `workers` CTAs (0: none)
__host__ __device__ inline int team_npt(int n, int sweeps, int workers)
{
    for (int npt = 4; npt <= 16; npt *= 2) {
        const int slab = kPT * npt - team_halo_left(sweeps) - kHaloR;
        if ((n + slab - 1) / slab <= workers) return npt;
    }
    return 0;
}

template <int NPT>
__device__ __noinline__ void big_visit(int l, int flags, int sweeps)
{
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const LevelConst& lc = g_sm.lc[l];
    const LevelConst& lcc = g_sm.lc[l + 1];
    const int n = lc.n;
    const int HL = team_halo_left(sweeps);
    const int slab = kPT * NPT - HL - kHaloR;
    const int wk = g_sm.team_rank - 1;
    const int a0 = wk * slab;
    if (a0 >= n) return;                                   // more workers than slabs
    const int b0 = min(a0 + slab, n);
    constexpr int W = kPT * NPT;                           // owned nodes of the window; node W is its fixed right end
    int wa = max(a0 - HL, 0);
    if (wa + W > n) wa = n - W;
    // window arrays in dynamic shared memory, node j at j + j / NPT (conflict-free per-thread chunks and coalesced copies)
    constexpr int WS = W + W / NPT + 2;
    double* phiL = g_dyn;
    double* srcL = g_dyn + WS;
    double* cL = g_dyn + 2 * WS;                           // coarse window (prolongation)
    const double* gp = g_sm.gphi + lc.op;
    const double* gs = g_sm.gsrc + lc.os;
    for (int j = t; j <= W; j += kPT) {
        const int sj = j + j / NPT;
        phiL[sj] = (flags & kLoadPhi) ? __ldcg(gp + wa + j) : 0.;
        srcL[sj] = __ldcg(gs + wa + j);
    }
    if (flags & kProlongIn) {
        const Ref Pc = Ref::P(l + 1);
        const Lay yc = lcc.lay;
        for (int q = t; q <= W / 2 + 1; q += kPT) cL[q] = Pc.ld(slot(min(wa / 2 + q, lcc.n), yc));
        __syncthreads();
        for (int j = t; j <= W; j += kPT) {
            const int sj = j + j / NPT;
            phiL[sj] += (j & 1) ? 0.5 * (cL[(j - 1) >> 1] + cL[(j + 1) >> 1]) : cL[j >> 1];
        }
    }
    __syncthreads();
    // sweeps: thread t owns window nodes [t NPT, (t+1) NPT); nodes 0 and W are fixed
    const double a = lc.a, bcoef = lc.bcoef;
    double phi[NPT], src[NPT];
#pragma unroll
    for (int k = 0; k < NPT; ++k) { phi[k] = phiL[t * (NPT + 1) + k]; src[k] = 0.5 * srcL[t * (NPT + 1) + k]; }
    const double right = phiL[W + W / NPT];
    double Ap[5];
    {
        double A = a;
#pragma unroll
        for (int k = 1; k < NPT; k <<= 1) A *= A;
        Ap[0] = A;
#pragma unroll
        for (int j = 1; j < 5; ++j) Ap[j] = Ap[j - 1] * Ap[j - 1];
    }
    const double B = Ap[4] * Ap[4];
    double Am[5];
    double Alane = 1.;
    int nsteps = 5;
#pragma unroll
    for (int j = 4; j >= 0; --j) if (Ap[j] < kTiny) nsteps = j;
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        Am[j] = (lane >= (1 << j) && j < nsteps) ? Ap[j] : 0.;
        if ((lane >> j) & 1) Alane *= Ap[j];
    }
    if (t == 0) g_sm.updates += (unsigned long long)sweeps * (unsigned long long)(b0 - a0);
    for (int sw = 0; sw < sweeps; ++sw) {
        double nb = __shfl_down_sync(full, phi[0], 1);
        if (lane == 0) g_sm.edge[w] = phi[0];
        __syncthreads();
        if (lane == 31 && w + 1 < (kPT >> 5)) nb = g_sm.edge[w + 1];
        if (t == kPT - 1) nb = right;
        double x = 0.;
#pragma unroll
        for (int k = 0; k < NPT; ++k) {
            const double c = fma(bcoef, (k + 1 < NPT) ? phi[k + 1] : nb, src[k]);
            x = (t == 0 && k == 0) ? phi[0] : fma(a, x, c);
            phi[k] = x;
        }
        double Pw = x;
        Pw = fma(Am[0], __shfl_up_sync(full, Pw, 1), Pw);
        if (nsteps > 1) {
            Pw = fma(Am[1], __shfl_up_sync(full, Pw, 2), Pw);
            if (nsteps > 2) {
                Pw = fma(Am[2], __shfl_up_sync(full, Pw, 4), Pw);
                Pw = fma(Am[3], __shfl_up_sync(full, Pw, 8), Pw);
                Pw = fma(Am[4], __shfl_up_sync(full, Pw, 16), Pw);
            }
        }
        if (lane == 31) g_sm.wtot[w] = Pw;
        __syncthreads();
        double carry = 0.;
        {
            double bp = 1.;
            for (int k = 1; k <= w && bp >= kTiny; ++k) { carry = fma(bp, g_sm.wtot[w - k], carry); bp *= B; }
        }
        double Pex = __shfl_up_sync(full, Pw, 1);
        if (lane == 0) Pex = 0.;
        double cin = fma(Alane, carry, Pex);
        if (t == 0) cin = 0.;
        double q = a;
#pragma unroll
        for (int k = 0; k < NPT; ++k) { phi[k] = fma(q, cin, phi[k]); q *= a; }
    }
#pragma unroll
    for (int k = 0; k < NPT; ++k) phiL[t * (NPT + 1) + k] = phi[k];
    __syncthreads();
    // the slab (and the right boundary node of the level, if it ends the slab) back to global memory
    double* gpw = g_sm.gphi + lc.op;
    for (int i = a0 + t; i < b0; i += kPT) { const int j = i - wa; gpw[i] = phiL[j + j / NPT]; }
    if (b0 == n && t == 0) gpw[n] = phiL[W + W / NPT];     // wa + W == n for the last slab
    if (flags & kRestrictOut) {
        const Ref Sc = Ref::S(l + 1);
        const Lay yc = lcc.lay;
        const double dc = lcc.d;
        for (int i = a0 / 2 + t; i < b0 / 2; i += kPT) {
            double v = 0.;
            if (i > 0) {
                const int j = 2 * i - wa;
                const double lft = phiL[(j - 1) + (j - 1) / NPT], mid = phiL[j + j / NPT], rgt = phiL[(j + 1) + (j + 1) / NPT];
                v = 4. * (srcL[j + j / NPT] + lft - 2. * mid + rgt) - dc * (rgt - lft);
            }
            Sc.st(slot(i, yc), v);
        }
        if (b0 == n && t == 0) Sc.st(lcc.n, 0.);
    }
    __syncthreads();
}

__device__ __noinline__ void big_visit_dispatch(int l, int flags, int sweeps)
{
    switch (team_npt(g_sm.lc[l].n, sweeps, g_sm.team_G - 1)) {
        case 4: big_visit<4>(l, flags, sweeps); break;
        case 8: big_visit<8>(l, flags, sweeps); break;
        default: big_visit<16>(l, flags, sweeps); break;
    }
}

// is level l run by a fused visit?  (single-chunk block levels and warp levels down to 64 nodes, all above the dense level m)
__device__ __forceinline__ bool fused_level(int l)
{
    const int n = g_sm.lc[l].n;
    return g_sm.has_G && l < g_sm.m && n <= kPT * kMaxNpt && n >= 64;
}
__device__ __noinline__ void fused_visit_block(int l, int flags, int sweeps)
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    switch (g_sm.lc[l].lay.lg) {
        case 5: fused_block<32, false>(l, flags, sweeps); break;
        case 4: fused_block<16, true>(l, flags, sweeps); break;
        case 3: fused_block<8, true>(l, flags, sweeps); break;
        case 2: fused_block<4, true>(l, flags, sweeps); break;
        default: fused_block<2, true>(l, flags, sweeps); break;
    }
    if (g_sm.dbg && threadIdx.x == 0) { g_sm.dbg[l] += clock64() - t0; g_sm.dbg[72 + l] += 1; }
}
__device__ __noinline__ void fused_visit_warp(int l, int flags, int sweeps)
{
    const long long t0 = g_sm.dbg ? clock64() : 0;
    switch (g_sm.lc[l].lay.lg) {
        case 4: fused_warp<16, true>(l, flags, sweeps); break;
        case 3: fused_warp<8, true>(l, flags, sweeps); break;
        case 2: fused_warp<4, true>(l, flags, sweeps); break;
        default: fused_warp<2, true>(l, flags, sweeps); break;
    }
    if (g_sm.dbg && threadIdx.x == 0) { g_sm.dbg[l] += clock64() - t0; g_sm.dbg[72 + l] += 1; }
}
// one level visit of a cycle, fused where possible, otherwise spelled out with the generic operators
__device__ __forceinline__ void visit(Ctl& ctl, int l, int flags, int sweeps)
{
    if (team_level(l)) {
        if (ctl.small_done) { block_begin(ctl); team_barrier(); ctl.small_done = false; }     // the leader's results become visible
        if (g_sm.team_rank > 0) big_visit_dispatch(l, flags, sweeps);
        team_barrier();
        return;
    }
    ctl.small_done = true;
    if (g_sm.team_rank > 0) return;                                                            // the leader's levels
    if (fused_level(l)) {
        if (g_sm.lc[l].wp == kWarp) {
            if (threadIdx.x < 32) fused_visit_warp(l, flags, sweeps);
            ctl.pending = true;
        } else {
            block_begin(ctl);
            fused_visit_block(l, flags, sweeps);
        }
        return;
    }
    // generic: the level arrays in memory are complete (Phi_l zeroed by the restriction that entered the level)
    if (flags & kProlongIn) prolong_from(ctl, l + 1);
    smooth(ctl, l, sweeps);
    if (flags & kRestrictOut) restrict_to(ctl, l + 1);
}
// The cycles  to_coarse(tops[q], c); to_fine(c, tops[q+1])  for the chain of top levels
//     first, first-1, ..., 1, 0, 0, ..., 0   (n_v times 0 -> 0 at the end),
// entered with Phi_first holding the result of the previous ascent (3 sweeps done) and left after the last ascent.
// Tops in the middle of the chain are one visit: prolong in, 3 + 3 sweeps, restrict out.
__device__ __noinline__ void cycle_chain(Ctl& ctl, int first, int n_v)
{
    const int m = g_sm.m;
    const int n_cycles = first + n_v;
    int a = first;
    bool top_done = false;               // the down-visit of level a was already part of the previous fused top
    for (int q = 0; q < n_cycles; ++q) {
        const int b = a > 0 ? a - 1 : 0;
        const bool last = (q == n_cycles - 1);
        for (int l = a; l < m; ++l) {
            if (l == a && top_done) continue;
            visit(ctl, l, (l == a ? kLoadPhi : 0) | kRestrictOut, 3);
        }
        if (g_sm.team_rank == 0) {
            if (threadIdx.x < 32) dense_apply_warp();
            ctl.pending = true;
        }
        for (int l = m - 1; l > b; --l) visit(ctl, l, kLoadPhi | kProlongIn, 3);
        if (last) { visit(ctl, b, kLoadPhi | kProlongIn, 3); top_done = false; }
        else { visit(ctl, b, kLoadPhi | kProlongIn | kRestrictOut, 6); top_done = true; }
        a = b;
    }
}

// natural order <-> owner-major order of level 0
__device__ __forceinline__ void import_level0(Ref dst, const double* nat, const double* scale, int N)
{
    const Lay y = g_sm.lc[0].lay;
    for (int s = threadIdx.x; s < N; s += blockDim.x) {
        const int i = unslot(s, y);
        dst.st(s, scale ? scale[i] * nat[i] : nat[i]);
    }
}
__device__ __forceinline__ void export_level0(double* nat, int N)
{
    const Lay y = g_sm.lc[0].lay;
    const Ref p = Ref::P(0);
    for (int s = threadIdx.x; s < N; s += blockDim.x) nat[unslot(s, y)] = p.ld(s);
}

// The same conversions for the 16385-node level 0 (512 threads x 32 nodes) with both sides coalesced: natural order <->
// padded natural order in dynamic shared memory (node i at i + i/32: a thread walking its own 32 nodes and a warp walking 32
// consecutive nodes are both conflict-free) <-> registers <-> owner-major slots.  The plain loops above gather 8-byte words
// 256 bytes apart (one 32-byte sector per word): measured ~10 % of a warm-started solve.  The staging area overlaps
// Source_0 and the start of the next shared level; it is only used before they are filled / after they are dead.
constexpr int kStageDoubles = kPT * kMaxNpt + kPT + 8;
__device__ __forceinline__ void stage_natural(const double* __restrict__ nat, const double* __restrict__ scale, int N)
{
    for (int i = threadIdx.x; i < N; i += kPT) g_dyn[i + (i >> 5)] = scale ? __ldg(scale + i) * __ldg(nat + i) : __ldg(nat + i);
    __syncthreads();
}
__device__ __forceinline__ void import_level0_staged(bool to_source, const double* __restrict__ nat, const double* __restrict__ scale, int N)
{
    const int t = threadIdx.x, n = N - 1;
    stage_natural(nat, scale, N);
    double v[kMaxNpt];
#pragma unroll
    for (int k = 0; k < kMaxNpt; ++k) v[k] = g_dyn[t * (kMaxNpt + 1) + k];
    const double vb = g_dyn[n + (n >> 5)];
    __syncthreads();
    const LevelConst& c = g_sm.lc[0];
    if (to_source) {                     // Source_0 lives in dynamic shared memory
#pragma unroll
        for (int k = 0; k < kMaxNpt; ++k) g_dyn[c.os + k * kPT + t] = v[k];
        if (t == 0) g_dyn[c.os + n] = vb;
    } else {                             // Phi_0 lives in global memory
        double* gp = g_sm.gphi + c.op;
#pragma unroll
        for (int k = 0; k < kMaxNpt; ++k) gp[k * kPT + t] = v[k];
        if (t == 0) gp[n] = vb;
    }
    __syncthreads();
}
__device__ __forceinline__ void export_level0_staged(double* __restrict__ nat, int N)
{
    const int t = threadIdx.x, n = N - 1;
    const double* gp = g_sm.gphi + g_sm.lc[0].op;
    __syncthreads();
    double v[kMaxNpt];
#pragma unroll
    for (int k = 0; k < kMaxNpt; ++k) v[k] = __ldcg(gp + k * kPT + t);
#pragma unroll
    for (int k = 0; k < kMaxNpt; ++k) g_dyn[t * (kMaxNpt + 1) + k] = v[k];
    if (t == 0) g_dyn[n + (n >> 5)] = __ldcg(gp + n);
    __syncthreads();
    for (int i = t; i < N; i += kPT) nat[i] = g_dyn[i + (i >> 5)];
}

// error-free transformations (Dekker / Knuth); the intrinsics keep nvcc from contracting or re-associating them
__device__ __forceinline__ void two_sum(double a, double b, double& s, double& e)
{
    s = __dadd_rn(a, b);
    const double bb = __dadd_rn(s, -a);
    e = __dadd_rn(__dadd_rn(a, -__dadd_rn(s, -bb)), __dadd_rn(b, -bb));
}
__device__ __forceinline__ void two_prod(double a, double b, double& p, double& e)
{
    p = __dmul_rn(a, b);
    e = __fma_rn(a, b, -p);
}
__device__ __forceinline__ void dd_add(double& hi, double& lo, double x, double xe)
{
    double s, e;
    two_sum(hi, x, s, e);
    hi = s;
    lo = __dadd_rn(lo, __dadd_rn(e, xe));
}

// residual of the fine-grid equation  U_{i-1}(1+δ/2) - 2 U_i + U_{i+1}(1-δ/2) = -S_i  in double-double.
// In FP64 the three U terms cancel to ~1e-7 of their size, which is what floors the plain iteration at ~1e-9 in U
// (SURVEY fact 3); evaluated with error-free transformations the residual is exact to ~1e-30.
__device__ __forceinline__ double dd_residual(double S, double um, double u0, double up, double cl, double cr)
{
    double hi = S, lo = 0., p, e;
    two_prod(cl, um, p, e); dd_add(hi, lo, p, e);
    dd_add(hi, lo, -2. * u0, 0.);
    two_prod(cr, up, p, e); dd_add(hi, lo, p, e);
    return __dadd_rn(hi, lo);
}

__global__ void __launch_bounds__(kPT) poisson_full_kernel(GridDev g, PoissonLevels lv, PoissonArgs a)
{
    const int G = a.team_G > 1 ? a.team_G : 1;          // CTAs per density (team mode: 1 leader + G - 1 workers)
    const int k = blockIdx.x / G, rank = blockIdx.x % G;
    const bool team = G > 1, leader = rank == 0;
    if (a.skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(a.skip) + (size_t)k * a.skip_stride_bytes)) return;
    const int N = g.N, L = lv.L, c = L - 1;
    const size_t NS = a.nat_stride ? (size_t)a.nat_stride : (size_t)N;       // row stride of the natural-order arrays
    const long long t_start = clock64();
    long long* dbg = (a.dbg && blockIdx.x == 0) ? a.dbg : nullptr;
    hierarchy_setup(lv, g.delta, a.phi + (size_t)k * lv.total, a.src + (size_t)k * lv.total, a.smem_doubles, a.coarse_op, dbg, G, rank,
                    team ? a.team_bar + k : nullptr);
    Ctl ctl{ false, false };
    const Ref phi = Ref::P(0), src = Ref::S(0);
    // team mode: level 0 is in natural node order in global memory, the workers split every pass over it
    const int ws0 = (rank - 1) * kPT + threadIdx.x, wstride = (G - 1) * kPT;

    // Source_0 (PoissonSolver.h:55-74)
    if (team) {
        if (!leader) {
            const double* rho = a.rho ? a.rho + (size_t)k * NS : a.src_nat + (size_t)k * NS;
            double* s0 = g_sm.gsrc + g_sm.lc[0].os;
            for (int i = ws0; i < N; i += wstride) s0[i] = a.rho ? g.psrc[i] * rho[i] : rho[i];
        }
    }
    const bool warm = a.warm_vcycles > 0 && a.u_out != nullptr;
    // 16385 nodes, one CTA: level 0 goes in and out through the staged (coalesced) conversions
    const bool staged_io = !team && N == kPT * kMaxNpt + 1 && g_sm.lc[0].ws == kDyn && g_sm.lc[0].wp == kGlobal && a.smem_doubles >= kStageDoubles;
    if (staged_io && warm) import_level0_staged(false, a.u_out + (size_t)k * NS, nullptr, N);       // (before Source_0: shares the staging area)
    if (!team) {
        if (staged_io && (a.rho || a.src_nat)) import_level0_staged(true, a.rho ? a.rho + (size_t)k * NS : a.src_nat + (size_t)k * NS, a.rho ? g.psrc : nullptr, N);
        else if (a.rho) import_level0(src, a.rho + (size_t)k * NS, g.psrc, N);
        else if (a.src_nat) import_level0(src, a.src_nat + (size_t)k * NS, nullptr, N);
    }
    const int n_cycles = warm ? a.warm_vcycles : a.max_vcycles;
    int fmg_top = 0;                     // top level the full-multigrid ramp has reached (0: only V-cycles are left)
    if (warm) {
        // Warm start (beyond the reference): Phi_0 = the previous solve of this density (u_out, same boundary values); the
        // V-cycles contract the difference by more than 10x each, so a few of them reach the same FP64 fixed point as the
        // full cycle from zero.  (Team mode: Phi_0 is still in place in global memory.)
        if (!team && !staged_io) import_level0(phi, a.u_out + (size_t)k * NS, nullptr, N);
        __syncthreads();
        team_barrier();
    } else {
        // Initialize (PoissonSolver.cpp:80-106) and the full-multigrid ramp (PoissonSolver.h:89-112)
        if (team) {
            if (!leader) { double* p0 = g_sm.gphi + g_sm.lc[0].op; for (int i = ws0; i < N; i += wstride) p0[i] = 0.; }
            team_barrier();
        } else {
            for (int s = threadIdx.x; s < N; s += blockDim.x) phi.st(s, 0.);
            __syncthreads();
        }
        for (int l = 1; l < L; ++l) {
            const Ref sf = Ref::S(l - 1), sc = Ref::S(l), pc = Ref::P(l);
            const int n = g_sm.lc[l].n + 1;
            const Lay yf = g_sm.lc[l - 1].lay, yc = g_sm.lc[l].lay;
            if (team_level(l)) {
                if (!leader)
                    for (int i = ws0; i < n; i += wstride) { sc.st(i, (i > 0 && i < n - 1) ? 4. * sf.ld(2 * i) : 0.); pc.st(i, 0.); }
                team_barrier();
            } else if (leader) {
                for (int s = threadIdx.x; s < n; s += blockDim.x) {
                    const int i = unslot(s, yc);
                    sc.st(s, (i > 0 && i < n - 1) ? 4. * sf.ld(slot(2 * i, yf)) : 0.);
                    pc.st(s, 0.);
                }
                __syncthreads();
            }
        }
        if (leader) {
            if (threadIdx.x == 0) {
                Ref::P(c).st(0, 0.);                                          // SetBoundaries(0, Z), PoissonSolver.h:76
                Ref::P(c).st(g_sm.lc[c].n, a.Zbc ? a.Zbc[k] : 0.);
            }
            __syncthreads();
            if (dbg && threadIdx.x == 0) dbg[98] += clock64() - t_start;
            smooth(ctl, c, 2);     // the coarsest level has one interior node: the reference's <= 15 sweeps converge in one
            // to_fine(c, l), to_coarse(l, c) for l = L-2 .. 1, then to_fine(c, 0)
            to_fine(ctl, c, L - 2);
        }
        fmg_top = L - 2;
    }
    const bool want_norm = (a.floor_stop || a.last_err) && a.u_out != nullptr;
    double* scratch = want_norm ? a.u_out + (size_t)k * NS : nullptr;      // overwritten by the export below
    double err = 0., prev = 1e300;
    int used = 0, stagnant = 0;
    // the ramp cycles whose top level is at or below the dense level are run level by level (the leader's levels)
    while (fmg_top > 0 && !(g_sm.has_G && fmg_top < g_sm.m)) { if (leader) cycle(ctl, fmg_top, fmg_top - 1, nullptr); --fmg_top; }
    ctl.small_done = true;
    if (g_sm.has_G && !want_norm) {
        cycle_chain(ctl, fmg_top, n_cycles);          // the rest of the ramp and the V-cycles, fused visits
        used = n_cycles;
    } else if (!team) {
        for (; fmg_top > 0; --fmg_top) cycle(ctl, fmg_top, fmg_top - 1, nullptr);
        for (int it = 0; it < n_cycles; ++it) {
            const bool last = (it == n_cycles - 1);
            ++used;
            if (want_norm && (last || a.floor_stop)) {
                err = cycle(ctl, 0, 0, scratch);
                if (err < 1e-14) break;                                   // PoissonSolver.h:120
                // the update norm contracts ~25x per cycle until it reaches its FP64 rounding floor (SURVEY fact 3)
                if (a.floor_stop) { if (err > 0.25 * prev) { if (++stagnant >= 2) break; } else stagnant = 0; }
                prev = err;
            } else {
                cycle(ctl, 0, 0, nullptr);
            }
        }
    }
    block_begin(ctl);
    // Defect correction (beyond the reference): one residual in double-double, then the error equation A e = r is solved
    // by the same V-cycles from e = 0 (its own rounding floor is ~1e-9 |e|, i.e. negligible) and U <- U + e.  The result
    // is the discrete solution to FP64 representation accuracy instead of ~1e-9, which removes the rounding-noise floor
    // of the SCF energies (the reference's |dE/E| wanders at 2e-11..1e-10 before it randomly dips below 1e-11).
    if (a.refine_vcycles > 0 && a.u0 && !team) {
        double* u0 = a.u0 + (size_t)k * NS;                            // slot order, like phi
        const double cl = 1. + 0.5 * g.delta, cr = 1. - 0.5 * g.delta;
        const Lay y0 = g_sm.lc[0].lay;
        // r into scratch, U0 saved, then Source_0 <- r, Phi_0 <- 0 (all levels' Phi are re-zeroed by restriction)
        for (int s = threadIdx.x; s < N; s += blockDim.x) {
            const int i = unslot(s, y0);
            u0[s] = (i > 0 && i < N - 1) ? dd_residual(src.ld(s), phi.ld(slot(i - 1, y0)), phi.ld(s), phi.ld(slot(i + 1, y0)), cl, cr) : 0.;
        }
        __syncthreads();
        for (int s = threadIdx.x; s < N; s += blockDim.x) {      // same thread owns slot s in both passes
            const double r = u0[s];
            u0[s] = phi.ld(s); src.st(s, r); phi.st(s, 0.);
        }
        __syncthreads();
        for (int it = 0; it < a.refine_vcycles; ++it) cycle(ctl, 0, 0, nullptr);
        block_begin(ctl);
        for (int s = threadIdx.x; s < N; s += blockDim.x) phi.st(s, phi.ld(s) + u0[s]);
        __syncthreads();
    }
    if (dbg && threadIdx.x == 0) dbg[96] += clock64() - t_start;
    if (team) {
        if (a.u_out && !leader) {
            const double* p0 = g_sm.gphi + g_sm.lc[0].op;
            double* u = a.u_out + (size_t)k * NS;
            for (int i = ws0; i < N; i += wstride) u[i] = __ldcg(p0 + i);
        }
    } else if (a.u_out) { if (staged_io) export_level0_staged(a.u_out + (size_t)k * NS, N); else export_level0(a.u_out + (size_t)k * NS, N); }
    if (dbg && threadIdx.x == 0) dbg[97] += clock64() - t_start;
    if (threadIdx.x == 0) {
        if (a.work) atomicAdd(a.work, g_sm.updates);
        if (leader && a.vcycles_used) a.vcycles_used[k] = used;
        if (leader && a.last_err) a.last_err[k] = err;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Dense operator of the coarse sub-cycle.  Thread j (1..31) runs the reference's sequence serially on the unit source
// e_j of the 32-node level m = L - 5:  [3 sweeps, restrict] down to the coarsest level, 3 sweeps there, [prolong,
// 3 sweeps] back up to level m (PoissonSolver.cpp:40-64, :110-157, :162-186), and stores the resulting Phi_m as
// column j.  Depends on (L, delta) only: built once per grid.
// ---------------------------------------------------------------------------------------------------------
__global__ void coarse_op_kernel(int L, double delta, double* G)
{
    const int j = threadIdx.x;
    double phi[6][33], src[6][33];          // levels m .. m+4 (32, 16, 8, 4, 2 owned nodes)
    const int m = L - 5;
    for (int q = 0; q < 6; ++q) for (int i = 0; i < 33; ++i) { phi[q][i] = 0.; src[q][i] = 0.; }
    if (j >= 1 && j < 32) src[0][j] = 1.;
    auto sweep3 = [&](int q) {
        const int n = 32 >> q;
        const double d = delta * (double)(1 << (m + q));
        const double a = 0.5 * (1. + 0.5 * d), b = 0.5 * (1. - 0.5 * d);
        for (int sw = 0; sw < 3; ++sw)
            for (int i = 1; i < n; ++i) phi[q][i] = fma(a, phi[q][i - 1], fma(b, phi[q][i + 1], 0.5 * src[q][i]));
    };
    for (int q = 0; q < 4; ++q) {
        sweep3(q);
        const int nc = 32 >> (q + 1);
        const double dc = delta * (double)(1 << (m + q + 1));
        for (int i = 0; i <= nc; ++i) {
            double v = 0.;
            if (i > 0 && i < nc) {
                const double lft = phi[q][2 * i - 1], mid = phi[q][2 * i], rgt = phi[q][2 * i + 1];
                v = 4. * (src[q][2 * i] + lft - 2. * mid + rgt) - dc * (rgt - lft);
            }
            phi[q + 1][i] = 0.;
            src[q + 1][i] = v;
        }
    }
    sweep3(4);
    for (int q = 4; q > 0; --q) {
        const int nc = 32 >> q;
        for (int i = 0; i <= nc; ++i) {
            const double c = phi[q][i];
            phi[q - 1][2 * i] += c;
            if (i > 0) phi[q - 1][2 * i - 1] += 0.5 * (phi[q][i - 1] + c);
        }
        sweep3(q - 1);
    }
    for (int i = 0; i < 32; ++i) G[j * 32 + i] = (j >= 1) ? phi[0][i] : 0.;
}

void launch_coarse_op(int L, double delta, double* G, cudaStream_t st)
{
    coarse_op_kernel<<<1, 32, 0, st>>>(L, delta, G);
}

// dynamic shared memory worth asking for: Source_0 plus every block level that fits (same greedy order as Hierarchy::setup)
static int dyn_doubles_for(const PoissonLevels& lv)
{
    const int cap = kMaxDynBytes / (int)sizeof(double);
    int avail = cap;
    const int n0 = lv.size[0] - 1;
    bool src0 = false;
    if (n0 > kWarpLevelNodes && ((n0 + 4) & ~3) <= avail) { src0 = true; avail -= (n0 + 4) & ~3; }
    for (int k = lv.L - 1; k >= 0; --k) {
        const int nk = lv.size[k] - 1;
        if (nk <= kWarpLevelNodes) continue;
        const int one = (nk + 4) & ~3;
        const int need = (k == 0 && src0) ? one : 2 * one;
        if (need > avail) break;
        avail -= need;
    }
    return cap - avail;
}

void launch_poisson_full(const GridDev& g, const PoissonLevels& lv, const PoissonArgs& a_in, cudaStream_t st)
{
    PoissonArgs a = a_in;
    a.smem_doubles = dyn_doubles_for(lv);
    size_t bytes = (size_t)a.smem_doubles * sizeof(double);
    // Team mode: large grids (levels above 16384 nodes) with so few densities that one CTA each would leave the GPU idle:
    // team_G CTAs per density, launched cooperatively (they synchronise through a per-density counter, so all of them must
    // be resident).  Needs the dense coarse operator (fused visits), no norm / refinement requests, and a barrier array.
    a.team_G = 1;
    const int n0 = lv.size[0] - 1;
    const int n_sm = a.n_sm > 0 ? a.n_sm : 148;
    if (n0 > kTeamLevelNodes && a.team_bar != nullptr && a.coarse_op != nullptr && !a.floor_stop && !a.last_err && a.refine_vcycles == 0) {
        const int G = std::min(41, n_sm / std::max(1, a.n_dens));
        if (G >= 2 && team_npt(n0, 6, G - 1) != 0) { a.team_G = G; bytes = kMaxDynBytes; }
    }
    if (a.team_G > 1) {
        cudaMemsetAsync(a.team_bar, 0, sizeof(unsigned) * a.n_dens, st);
        GridDev gg = g; PoissonLevels ll = lv;
        void* args[] = { &gg, &ll, &a };
        cudaLaunchCooperativeKernel((const void*)poisson_full_kernel, dim3(a.n_dens * a.team_G), dim3(kPT), args, bytes, st);
    } else {
        poisson_full_kernel<<<a.n_dens, kPT, bytes, st>>>(g, lv, a);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Stream mode (many densities on a grid that does not fit on chip, poisson_stream.cu): the levels above 16384 nodes are
// visited by stream_visit_kernel launches over all densities; this kernel is the part of the V-cycle below them, one CTA
// per density: it takes Source_K (K = the 16384-node level, natural node order, written by the restriction of level K-1),
// runs  visit(K) ... restrict ... dense coarse operator ... prolong ... visit(K)  with Phi_K starting from zero, and leaves
// Phi_K in natural order for the prolongation into level K-1.  Its own level arrays (owner-major) live in mid_phi/mid_src.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kPT) poisson_mid_kernel(double delta, PoissonLevels lv, int K, double* nat_phi, const double* nat_src,
                                                         long long nat_stride, double* mid_phi, double* mid_src, int mid_total,
                                                         const double* Gg, int smem_doubles, const int* skip, int skip_stride_bytes)
{
    const int k = blockIdx.x;
    if (skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(skip) + (size_t)k * skip_stride_bytes)) return;
    // (the level offsets of `lv` count from level 0: shift the block so that level K lands at its start)
    hierarchy_setup(lv, delta, mid_phi + (size_t)k * mid_total - lv.off[K], mid_src + (size_t)k * mid_total - lv.off[K], smem_doubles, Gg,
                    nullptr, 2, 0, nullptr);
    const int nK = g_sm.lc[K].n, m = g_sm.m;
    const Lay yK = g_sm.lc[K].lay;
    const Ref SK = Ref::S(K), PK = Ref::P(K);
    const double* ns = nat_src + (size_t)k * nat_stride;
    double* np = nat_phi + (size_t)k * nat_stride;
    for (int i = threadIdx.x; i <= nK; i += blockDim.x) SK.st(slot(i, yK), __ldcg(ns + i));
    __syncthreads();
    Ctl ctl{ false, false };
    for (int l = K; l < m; ++l) visit(ctl, l, kRestrictOut, 3);
    if (threadIdx.x < 32) dense_apply_warp();
    ctl.pending = true;
    for (int l = m - 1; l >= K; --l) visit(ctl, l, kLoadPhi | kProlongIn, 3);
    block_begin(ctl);
    __syncthreads();
    for (int i = threadIdx.x; i <= nK; i += blockDim.x) np[i] = PK.ld(slot(i, yK));
}

void launch_poisson_mid(const PoissonLevels& lv, double delta, int K, int n_dens, double* nat_phi, const double* nat_src, long long nat_stride,
                        double* mid_phi, double* mid_src, int mid_total, const double* coarse_op, const int* skip, int skip_stride_bytes,
                        cudaStream_t st)
{
    const int sd = dyn_doubles_for(lv);
    const size_t bytes = (size_t)sd * sizeof(double);
    poisson_mid_kernel<<<n_dens, kPT, bytes, st>>>(delta, lv, K, nat_phi, nat_src, nat_stride, mid_phi, mid_src, mid_total, coarse_op, sd, skip, skip_stride_bytes);
}

// V-cycles as defined by the reference on given (Phi_0, Source_0) in natural node order: parity / microbench entry point
// (every level is swept level by level: no dense coarse operator)
__global__ void __launch_bounds__(kPT) poisson_vcycles_kernel(double delta, PoissonLevels lv, double* phi_all, double* src_all,
                                                             double* phi_nat, const double* src_nat, int smem_doubles, int n_cycles,
                                                             double* last_err)
{
    const int k = blockIdx.x;
    const int N = lv.size[0];
    hierarchy_setup(lv, delta, phi_all + (size_t)k * lv.total, src_all + (size_t)k * lv.total, smem_doubles, nullptr, nullptr);
    Ctl ctl{ false, false };
    import_level0(Ref::P(0), phi_nat + (size_t)k * N, nullptr, N);
    import_level0(Ref::S(0), src_nat + (size_t)k * N, nullptr, N);
    __syncthreads();
    double err = 0.;
    for (int it = 0; it < n_cycles; ++it) err = cycle(ctl, 0, 0, it == n_cycles - 1 ? phi_nat + (size_t)k * N : nullptr);
    block_begin(ctl);
    export_level0(phi_nat + (size_t)k * N, N);
    if (threadIdx.x == 0 && last_err) last_err[k] = err;
}

void launch_poisson_vcycles(const PoissonLevels& lv, double delta, int n_dens, double* phi, double* src, double* phi_nat,
                            const double* src_nat, int n_cycles, double* last_err, cudaStream_t st)
{
    const int sd = dyn_doubles_for(lv);
    const size_t bytes = (size_t)sd * sizeof(double);
    poisson_vcycles_kernel<<<n_dens, kPT, bytes, st>>>(delta, lv, phi, src, phi_nat, src_nat, sd, n_cycles, last_err);
}

// per-device opt-in to the dynamic shared memory the solve kernels may ask for (called from dftatom_create under cudaSetDevice)
int poisson_init_device()
{
    DFT_CHECK(cudaFuncSetAttribute(poisson_full_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynBytes));
    DFT_CHECK(cudaFuncSetAttribute(poisson_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynBytes));
    DFT_CHECK(cudaFuncSetAttribute(poisson_vcycles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynBytes));
    return 0;
}

}  // namespace dft
