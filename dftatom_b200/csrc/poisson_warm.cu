// Warm-started radial Poisson V-cycles in increment form for grids of 2049 .. 16385 nodes: ONE CTA (one SM) PER DENSITY.
//
// Replaces (reference DFTAtom/) PoissonSolver.h:155-159 VCycle, PoissonSolver.cpp:40-64 GaussSeidel, :110-123 Prolong, :126-157 Restrict,
// :162-197 Ascend / Descend for the warm solves of the SCF: from SCF step `warm_after` on a solve is `warm_vcycles` V-cycles on
//   A dU = -r 4 pi K (rho - rho_prev),  dU = 0 on both boundaries and as the initial guess,  U += dU        (scf.cu: increment form).
// Same operators and the same order of sweeps / restriction / prolongation as poisson.cu.  What this kernel is built around: a solve is a
// chain of dependent Gauss-Seidel sweeps and level visits, each only a few hundred cycles of work for one SM.
//  * Every level is visited by the whole CTA: thread t owns NPT = n / 512 consecutive nodes (one node per thread on the first n threads
//    below 512 nodes).  A visit loads them into registers ONCE, (adds the prolongated correction,) runs its 3 or 6 sweeps on the
//    registers, (forms the restricted residual of the next level,) and stores once.  Where a level lives is a template parameter: no
//    generic loads, no per-element branches, every transfer of a visit is one batch of independent loads.
//  * A sweep is the zero-carry local recurrence Phi_i = a Phi_{i-1} + (b Phi_{i+1} + S_i/2), a truncated warp scan of the affine maps
//    (a ~ 1/2: a^64 < 1e-19) and the carry patch - with ONE block barrier: the right neighbour warp's old first node and the left
//    neighbour warp's total are published before it (double buffered by sweep parity); what lane 31 could not know before the barrier
//    (b x the neighbour's first node) is added to its last node and to the carry of the next warp after it.
//  * The levels below 2048 nodes are replaced by the exact solve of the 1024-node level (poisson_tri.cuh).
//  * Source_0/2 and the levels of <= 2048 nodes live in shared memory (owner-major: thread t's k-th node at k x 513 + t, conflict-free both
//    for the owner and for the coalesced import / export), Phi_0 and the two levels of 8192 / 4096 nodes in this density's block of the
//    L2-resident hierarchy buffers (owner-major, coalesced): ~0.9 MB of L2 traffic per V-cycle and density.
#include "internal.h"
#include "poisson_tri.cuh"
#include <algorithm>
#include <cmath>
#include <cstdio>

namespace dft {
namespace {

constexpr int kWT = 512;             // threads per CTA
constexpr int kWStride = kWT + 1;    // owner-major stride of the block levels in shared memory
constexpr double kTinyW = 1e-19;
enum { kWLoad = 1, kWProlong = 2, kWRestrict = 4, kWExport = 8 };

struct WLevel {
    int n;                  // owned nodes 0 .. n-1 (node 0 is the left boundary, pinned to 0); node n is the right boundary (0)
    int npt;                // nodes per owner; owners = n / npt = min(n, 512)
    int gl;                 // 1: Phi (and, below level 0, Source / 2) in the global blocks; 0: shared memory
    int offP, offS;         // element (owner o, k) of Phi at offP + k strideP + o, of Source / 2 at offS + k strideS + o
    int strideP, strideS;
    int nsteps;             // warp-scan steps that still matter
    double d, a, b;         // d_l = delta 2^l; a = (1 + d/2)/2; b = (1 - d/2)/2       (PoissonSolver.cpp:56-57)
    double Ap[5], B;        // A^(2^j), A = a^npt (one owner's affine map); A^32 (one warp)
    double apow[32];        // a^(k+1): the carry patch of an owner's k-th node
    double alane[32];       // A^lane
};

struct WShared {
    WLevel lv[12];
    int m;                  // the exactly solved 1024-node level
    int offT;               // its table in w_dyn
    double* gphi; double* gsrc;     // this density's blocks of the global hierarchy buffers
    double* U;
    double edge[2][kWT / 32 + 1];   // old first node of every warp, by sweep parity
    double wtot[2][kWT / 32];       // scan total of every warp (without b x the right neighbour's first node)
    double last[kWT / 32];          // last node of every warp after the sweeps (restriction)
    unsigned long long updates;
#ifdef DFT_WARM_DEBUG
    long long clk[64];
#endif
};
__shared__ WShared ws;
extern __shared__ double w_dyn[];

#ifdef DFT_WARM_DEBUG
__device__ long long g_warm_clk[64];
#define WCLK(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); ws.clk[40 + (i)] += t_ - tw; tw = t_; } } while (0)
#else
#define WCLK(i) do { } while (0)
#endif

// The sweeps of a visit on an owner's registers.  Source / 2 of the owner's nodes: registers (SREG) or a shared-memory row (srow).
template <int NPT, bool SREG>
__device__ __forceinline__ void w_sweeps(double (&phi)[NPT], const double (&hs)[SREG ? NPT : 1], const double* __restrict__ srow, int strideS,
                                         const WLevel& c, int sweeps, int o, int owners, bool active)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double a = c.a, b = c.b;
    const int nsteps = c.nsteps;
    const double B = c.B;
    const int nwarps = owners >> 5;
    const double Am0 = (lane >= 1 && nsteps > 0) ? c.Ap[0] : 0.;     // (the multipliers of the later steps are read where they are used: registers)
    const double Alane = c.alane[lane];
    constexpr int NAP = NPT <= 8 ? NPT : 1;
    double ap[NAP];
#pragma unroll
    for (int k = 0; k < NAP; ++k) ap[k] = c.apow[k];
    int par = 0;
    for (int sw = 0; sw < sweeps; ++sw) {
        double P = 0., e0 = 0.;
        if (active) {
            e0 = phi[0];
            if (lane == 0) ws.edge[par][w] = e0;
        }
        double nb = __shfl_down_sync(full, e0, 1);
        if (lane == 31) nb = 0.;                // the right neighbour warp's first node follows after the barrier; last owner: Phi_n = 0
        if (active) {
            // local recurrence with zero carry-in, in place
            double x = 0.;
            if (SREG) {
#pragma unroll
                for (int k = 0; k < NPT; ++k) {
                    const double cc = fma(b, (k + 1 < NPT) ? phi[k + 1] : nb, hs[SREG ? k : 0]);
                    x = fma(a, x, cc);
                    if (k == 0 && o == 0) x = 0.;   // node 0 is the left boundary
                    phi[k] = x;
                }
            } else {
                // Source / 2 from shared memory: the b Phi_{i+1} + S_i/2 terms of 8 nodes first (independent), then their chain
                constexpr int CH = NPT < 4 ? NPT : 4;
#pragma unroll
                for (int k0 = 0; k0 < NPT; k0 += CH) {
                    double cc[CH];
#pragma unroll
                    for (int q = 0; q < CH; ++q) { const int k = k0 + q; cc[q] = fma(b, (k + 1 < NPT) ? phi[k + 1] : nb, srow[k * strideS]); }
#pragma unroll
                    for (int q = 0; q < CH; ++q) {
                        x = fma(a, x, cc[q]);
                        if (k0 + q == 0 && o == 0) x = 0.;
                        phi[k0 + q] = x;
                    }
                }
            }
            P = x;
        }
        // warp scan of the totals (uniform multiplier A = a^NPT): P_lane = sum_j A^(lane-j) x_j, truncated where A^(2^j) < 1e-19
        P = fma(Am0, __shfl_up_sync(full, P, 1), P);
        if (nsteps > 1) {
            P = fma(lane >= 2 ? c.Ap[1] : 0., __shfl_up_sync(full, P, 2), P);
            if (nsteps > 2) {
                P = fma(lane >= 4 ? c.Ap[2] : 0., __shfl_up_sync(full, P, 4), P);
                if (nsteps > 3) {
                    P = fma(lane >= 8 ? c.Ap[3] : 0., __shfl_up_sync(full, P, 8), P);
                    P = fma((lane >= 16 && nsteps > 4) ? c.Ap[4] : 0., __shfl_up_sync(full, P, 16), P);
                }
            }
        }
        if (active && lane == 31) ws.wtot[par][w] = P;
        __syncthreads();
        double Pex = __shfl_up_sync(full, P, 1);
        const double e0w = __shfl_sync(full, e0, 0);
        if (active) {
            double carry = 0., fix = 0.;
            if (lane == 31 && w + 1 < nwarps) fix = b * ws.edge[par][w + 1];
            if (w > 0) {
                // new value of the node left of this warp: sum_k B^(k-1) (W_(w-k) + b e_(w-k+1)), truncated
                carry = fma(b, e0w, ws.wtot[par][w - 1]);
                double bp = B;
                for (int k = 2; k <= w && bp >= kTinyW; ++k) { carry = fma(bp, fma(b, ws.edge[par][w - k + 1], ws.wtot[par][w - k]), carry); bp *= B; }
            }
            if (lane == 0) Pex = 0.;
            double cin = fma(Alane, carry, Pex);    // new value of the node before this owner's first node
            if (o == 0) cin = 0.;
#pragma unroll
            for (int k = 0; k < NPT; ++k) phi[k] = fma(NPT <= 8 ? ap[k < NAP ? k : 0] : c.apow[k], cin, phi[k]);
            if (lane == 31) phi[NPT - 1] += fix;
        }
        par ^= 1;
    }
}

// One level visit.  Template: nodes per owner; PG / SG: Phi / Source of THIS level in the global blocks (else shared memory); CG: both arrays
// of the NEXT (coarser) level in the global blocks.  NPT >= 2: the coarse nodes of an owner's fine nodes are its own (same owner index);
// NPT == 1: coarse node i is owned by thread i, the transfers go through shared memory.
__device__ __forceinline__ int w_tri_addr(int i) { return (i >> 5) * 33 + (i & 31); }       // layout of the exactly solved level: lane-major rows of 33

template <int NPT, bool PG, bool SG, bool CG, bool CT = false>
__device__ __noinline__ void w_visit(int l, int flags, int sweeps)
{
    const unsigned full = 0xffffffffu;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const WLevel& c = ws.lv[l];
    const int owners = c.n / NPT;
    const bool active = t < owners;
    const int o = t;
    double* const Pp = (PG ? ws.gphi : w_dyn) + c.offP + o;
    const double* const Sp = (SG ? ws.gsrc : w_dyn) + c.offS + o;
    const int strideP = c.strideP, strideS = c.strideS;
    constexpr bool SREG = NPT <= 16;
    constexpr int NC = NPT >= 2 ? NPT / 2 : 1;
    double phi[NPT], hs[SREG ? NPT : 1];
#ifdef DFT_WARM_DEBUG
    long long tw = clock64();
#endif
    __syncthreads();                            // what the previous visit stored (and its reads of edge / wtot / last) is behind us
#pragma unroll
    for (int k = 0; k < NPT; ++k) phi[k] = 0.;
#pragma unroll
    for (int k = 0; k < (SREG ? NPT : 1); ++k) hs[k] = 0.;
    if (active) {
        if (flags & kWLoad) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) phi[k] = Pp[k * strideP];
        }
        if (SREG) {
#pragma unroll
            for (int k = 0; k < NPT; ++k) hs[SREG ? k : 0] = Sp[k * strideS];
        }
    }
    WCLK(0);
    if ((flags & kWProlong) && active) {        // Phi_l += P Phi_{l+1}   (PoissonSolver.cpp:110-123)
        const WLevel& cc = ws.lv[l + 1];
        const double* const Cb = (CG ? ws.gphi : w_dyn) + cc.offP;
        if (NPT >= 2) {
            // coarse nodes o NC .. o NC + NC: the owner's own and the first one of the next owner (the right boundary, 0, behind the last owner)
            const int strideC = cc.strideP;
            double cprev = CT ? Cb[w_tri_addr(o * NC)] : Cb[o];
            phi[0] += cprev;
#pragma unroll
            for (int j = 1; j <= NC; ++j) {
                const double cj = CT ? ((j < NC || o + 1 < owners) ? Cb[w_tri_addr(o * NC + j)] : 0.)
                                     : (j < NC ? Cb[j * strideC + o] : ((o + 1 < owners) ? Cb[o + 1] : 0.));
                phi[2 * j - 1] += 0.5 * (cprev + cj);
                if (2 * j < NPT) phi[2 * j < NPT ? 2 * j : 0] += cj;
                cprev = cj;
            }
        } else {
            // one node per thread on both levels (natural order)
            const int i0 = o >> 1, i1 = (o + 1) >> 1;
            const double c0 = Cb[i0], c1 = (i1 < cc.n) ? Cb[i1] : 0.;
            phi[0] += (o & 1) ? 0.5 * (c0 + c1) : c0;
        }
        if (o == 0) phi[0] = 0.;
    }
    WCLK(1);
    w_sweeps<NPT, SREG>(phi, hs, Sp, strideS, c, sweeps, o, owners, active);
    WCLK(2);
    if (t == 0 && !(flags & kWExport)) ws.updates += (unsigned long long)sweeps * (unsigned long long)c.n;
    if (flags & kWExport) {                     // U += dU: through shared memory (the Source_0 rows) for coalesced global accesses
        __syncthreads();                        // every thread is done with Source_0
        double* const T = w_dyn + c.offS + o;
#pragma unroll
        for (int k = 0; k < NPT; ++k) T[k * strideS] = phi[k];
        __syncthreads();
        for (int i = t; i < c.n; i += kWT) ws.U[i] += w_dyn[c.offS + (i % NPT) * strideS + i / NPT];
        return;
    }
    if (active) {
#pragma unroll
        for (int k = 0; k < NPT; ++k) Pp[k * strideP] = phi[k];
    }
    if (flags & kWRestrict) {                   // Source_{l+1} = R (Source_l - A Phi_l)   (PoissonSolver.cpp:126-157), stored halved; Phi_{l+1} starts from 0
        const WLevel& cc = ws.lv[l + 1];
        double* const CS = (CG ? ws.gsrc : w_dyn) + cc.offS;
        const double dc = cc.d;
        if (NPT >= 2) {
            double prev = __shfl_up_sync(full, phi[NPT - 1], 1);
            if (lane == 31) ws.last[w] = phi[NPT - 1];
            __syncthreads();
            if (lane == 0 && w > 0) prev = ws.last[w - 1];
            if (active) {
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                    const double lft = j ? phi[2 * j - 1 >= 0 ? 2 * j - 1 : 0] : prev, mid = phi[2 * j < NPT ? 2 * j : 0], rgt = phi[2 * j + 1 < NPT ? 2 * j + 1 : 0];
                    const double S = 2. * (SREG ? hs[(SREG && 2 * j < NPT) ? 2 * j : 0] : Sp[2 * j * strideS]);
                    const double v = 4. * (S + lft - 2. * mid + rgt) - dc * (rgt - lft);
                    CS[CT ? w_tri_addr(o * NC + j) : j * cc.strideS + o] = (o == 0 && j == 0) ? 0. : 0.5 * v;
                }
            }
        } else {
            // one node per thread: the fine values through shared memory (this level's Phi was just stored there)
            __syncthreads();
            if (t < cc.n) {
                const double* const Pf = w_dyn + c.offP;
                const double lft = t ? Pf[2 * t - 1] : 0., mid = Pf[2 * t], rgt = Pf[2 * t + 1];
                const double S = 2. * (w_dyn + c.offS)[2 * t];
                const double v = 4. * (S + lft - 2. * mid + rgt) - dc * (rgt - lft);
                CS[t] = t ? 0.5 * v : 0.;
            }
        }
    }
    WCLK(3);
}

__device__ __forceinline__ void w_visit_level_impl(int l, int flags, int sweeps)
{
    const WLevel& c = ws.lv[l];
    const bool cg = ws.lv[l + 1].gl != 0;
    const bool ct = l + 1 == ws.m;              // the next level is the exactly solved one
    if (l == 0) {               // Phi_0 in the global block, Source_0 / 2 in shared memory
        switch (c.npt) {
            case 32: w_visit<32, true, false, true>(l, flags, sweeps); break;
            case 16: w_visit<16, true, false, true>(l, flags, sweeps); break;
            case 8: w_visit<8, true, false, false>(l, flags, sweeps); break;
            default: if (ct) w_visit<4, true, false, false, true>(l, flags, sweeps); else w_visit<4, true, false, false>(l, flags, sweeps); break;
        }
    } else if (c.gl) {          // 8192 / 4096 nodes below level 0
        if (c.npt == 16) w_visit<16, true, true, true>(l, flags, sweeps);
        else if (cg) w_visit<8, true, true, true>(l, flags, sweeps);
        else w_visit<8, true, true, false>(l, flags, sweeps);
    } else {
        switch (c.npt) {
            case 4: if (ct) w_visit<4, false, false, false, true>(l, flags, sweeps); else w_visit<4, false, false, false>(l, flags, sweeps); break;
            case 2: w_visit<2, false, false, false>(l, flags, sweeps); break;
            default: w_visit<1, false, false, false>(l, flags, sweeps); break;
        }
    }
}
__device__ __forceinline__ void w_visit_level(int l, int flags, int sweeps)
{
#ifdef DFT_WARM_DEBUG
    const long long t0 = clock64();
    w_visit_level_impl(l, flags, sweeps);
    if (threadIdx.x == 0) ws.clk[l + ((flags & kWLoad) ? 16 : 0)] += clock64() - t0;
#else
    w_visit_level_impl(l, flags, sweeps);
#endif
}

// exact solve of the 1024-node level (warp 0), in place of everything below the 2048-node level
__device__ __forceinline__ void w_tri()
{
    __syncthreads();
    if (threadIdx.x < 32) {
        const WLevel& c = ws.lv[ws.m];
        const double* hS = w_dyn + c.offS;
        double* P = w_dyn + c.offP;
        tri_solve_warp(w_dyn + ws.offT, c.a, c.b, [&](int i) { return hS[w_tri_addr(i)]; }, [&](int i, double v) { P[w_tri_addr(i)] = v; });
    }
}

// placement of the levels 0 .. L-10.  Phi_0 and both arrays of the levels of >= 4096 nodes below it live in the global blocks (stride 512),
// everything else in shared memory (stride 513 with 512 owners; natural order below)
__host__ __device__ inline void w_place_all(int L, WLevel* out, int& dyn, int& gph, int& gsr, int& offT)
{
    dyn = 0; gph = 0; gsr = 0; offT = 0;
    const int last = L - 10;
    for (int q = 0; q <= last; ++q) {
        const int n = 1 << (L - q);
        if (q == last) {                // the exactly solved level: lane-major rows of 33, and its table
            const int offP = dyn, offS = dyn + 32 * 33 + 1;
            dyn += 2 * (32 * 33 + 1);
            offT = dyn; dyn += kTriTableDoubles;
            if (out) { WLevel& c = out[q]; c.n = n; c.npt = 2; c.gl = 0; c.offP = offP; c.offS = offS; c.strideP = 0; c.strideS = 0; }
            break;
        }
        const int npt = n >= kWT ? n / kWT : 1;
        const int owners = n / npt;
        const int gl = (q == 0 || n >= 4096) ? 1 : 0;
        const bool gS = gl && q > 0;
        const int strideP = gl ? kWT : (owners == kWT ? kWStride : owners);
        const int strideS = gS ? kWT : (owners == kWT ? kWStride : owners);
        int offP, offS;
        if (gl) { offP = gph; gph += npt * kWT; } else { offP = dyn; dyn += npt * strideP + 2; }
        if (gS) { offS = gsr; gsr += npt * kWT; } else { offS = dyn; dyn += npt * strideS + 2; }
        if (out) { WLevel& c = out[q]; c.n = n; c.npt = npt; c.gl = gl; c.offP = offP; c.offS = offS; c.strideP = strideP; c.strideS = strideS; }
    }
}

}  // namespace

__global__ void __launch_bounds__(kWT, 1) poisson_warm_kernel(GridDev g, WarmPoissonArgs a, double* gphi_all, double* gsrc_all, long long gstride)
{
    const int k = blockIdx.x;
    if (a.skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(a.skip) + (size_t)k * a.skip_stride_bytes)) return;
    const int L = g.L, N = g.N, t = threadIdx.x;
    const int m = L - 10;
    if (t == 0) {
        int dyn, gph, gsr, offT;
        w_place_all(L, ws.lv, dyn, gph, gsr, offT);
        ws.lv[m + 1].gl = 0;
        ws.m = m; ws.offT = offT;
        ws.gphi = gphi_all + (size_t)k * gstride; ws.gsrc = gsrc_all + (size_t)k * gstride;
        ws.U = a.U + (size_t)k * a.ldU;
        ws.updates = 0;
#ifdef DFT_WARM_DEBUG
        for (int q = 0; q < 64; ++q) ws.clk[q] = 0;
#endif
    }
    __syncthreads();
    if (t <= m) {
        WLevel& c = ws.lv[t];
        c.d = g.delta * (double)(1 << t);
        c.a = 0.5 * (1. + 0.5 * c.d);
        c.b = 0.5 * (1. - 0.5 * c.d);
        double q = c.a;
        for (int e = 0; e < 32; ++e) { c.apow[e] = q; q *= c.a; }
        c.Ap[0] = c.apow[c.npt - 1];
        for (int j = 1; j < 5; ++j) c.Ap[j] = c.Ap[j - 1] * c.Ap[j - 1];
        c.B = c.Ap[4] * c.Ap[4];
        c.nsteps = 5;
        for (int j = 4; j >= 0; --j) if (c.Ap[j] < kTinyW) c.nsteps = j;
        for (int ln = 0; ln < 32; ++ln) {
            double al = 1.;
            for (int j = 0; j < 5; ++j) if ((ln >> j) & 1) al *= c.Ap[j];
            c.alane[ln] = al;
        }
    }
    for (int i = t; i < kTriTableDoubles; i += kWT) w_dyn[ws.offT + i] = a.coarse_tri[i];
    __syncthreads();
    // import: Source_0 / 2 = r 4 pi K (rho - rho_prev) / 2 into its owner-major rows; rho_prev = rho
    {
        const WLevel& c0 = ws.lv[0];
        const double* rho = a.rho + (size_t)k * a.rho_stride;
        double* rp = a.rho_prev + (size_t)k * a.rho_stride;
        const int npt0 = c0.npt;
        for (int i = t; i < N; i += kWT) {
            const double r = rho[i];
            const double base = rp[i];
            if (i < c0.n) w_dyn[c0.offS + (i % npt0) * c0.strideS + i / npt0] = (i >= 1) ? 0.5 * (g.psrc[i] * (r - base)) : 0.;
            rp[i] = r;
        }
    }
    const int nv = a.n_vcycles;
    for (int cyc = 0; cyc < nv; ++cyc) {
        // down-leg (the level-0 down-visit of every cycle but the first was fused into the previous top); dU starts from 0
        for (int l = (cyc == 0 ? 0 : 1); l < m; ++l) w_visit_level(l, kWRestrict, 3);
        w_tri();
        // up-leg
        for (int l = m - 1; l >= 1; --l) w_visit_level(l, kWLoad | kWProlong, 3);
        if (cyc == nv - 1) w_visit_level(0, kWLoad | kWProlong | kWExport, 3);
        else w_visit_level(0, kWLoad | kWProlong | kWRestrict, 6);
    }
    if (t == 0 && a.work) atomicAdd(a.work, ws.updates);
#ifdef DFT_WARM_DEBUG
    if (t == 0 && k == 0 && g_warm_clk[0]++ % 40 == 0) {
        printf("warm clk of one solve per level (down | up):");
        for (int l = 0; l <= m; ++l) printf(" [%d] %lld | %lld", l, ws.clk[l], ws.clk[16 + l]);
        printf("\n   phases: sync+load %lld prolong %lld sweeps %lld store+restrict %lld\n", ws.clk[40], ws.clk[41], ws.clk[42], ws.clk[43]);
    }
#endif
}

static int warm_smem_doubles(int L)
{
    int dyn, gph, gsr, offT;
    w_place_all(L, nullptr, dyn, gph, gsr, offT);
    return dyn;
}

// table of the exact solve of the 1024-node level of an L-level grid (poisson_tri.cuh), kTriTableDoubles doubles; built on the host once per grid
void coarse_tri_host(int L, double delta, double* T) { tri_build_table(delta * (double)(1 << (L - 10)), T); }

bool poisson_warm_supported(int L, double delta) { return L >= 11 && L <= 14 && delta > 0.; }

long long poisson_warm_scratch_doubles(int L)
{
    int dyn, gph, gsr, offT;
    w_place_all(L, nullptr, dyn, gph, gsr, offT);
    return std::max(gph, gsr);
}

int poisson_warm_init_device()
{
    DFT_CHECK(cudaFuncSetAttribute(poisson_warm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, warm_smem_doubles(14) * (int)sizeof(double)));
    return 0;
}

// a: a.coarse_tri required; gphi / gsrc: two scratch buffers of n_dens x gstride doubles, gstride >= poisson_warm_scratch_doubles(L)
void launch_poisson_warm(const GridDev& g, const WarmPoissonArgs& a, double* gphi, double* gsrc, long long gstride, cudaStream_t st)
{
    poisson_warm_kernel<<<a.n_dens, kWT, (size_t)warm_smem_doubles(g.L) * sizeof(double), st>>>(g, a, gphi, gsrc, gstride);
}

}  // namespace dft
