// Numerov shooting with the radial grid across the lanes ("rows" kernel): the production energy search of one level.
//
// Replaces the same reference code as numerov_seg.cu / numerov_fast.cu (DFTAtom.cpp:493-541, :566-604; Numerov.h:272-401) with the same
// monotone search predicate (numerov_common.cuh) and the same recurrence (numerov_sweep.cuh), but turned by 90 degrees:
//   numerov_seg.cu  : lane = trial energy (32 per round), warp = radial segment, cluster of CTAs per orbital, 3 cluster barriers per round;
//   this file       : lane = radial segment, every thread carries kRowE = 4 trial energies x 2 basis chains in registers (8 independent
//                     dependence chains: a lone warp keeps its FP64 pipe busy), ONE CTA of 4 warps per orbital, no cluster, block barriers only.
// A round costs (trial energies) x (nodes) x 11 FP64 instructions whatever the shape, so what the shape decides is how many trial
// energies a solve needs and how deep the dependent chain of a round is.  With 32 energies per round a solve took 2.2-2.5 rounds = 70-80
// sweeps; y0(E) is smooth, so once the root is bracketed by four samples the inverse cubic interpolation is good to ~1e-12 and a round of
// FOUR energies (two at +-0.45 energyErr around the estimate, two at the trust radius) closes the bracket: 8 + 4 (+ 4) sweeps per solve.
// The 4 warps of the CTA are dealt per round as NG energy groups x SW sub-warps (NG x SW = 4): 16 energies x 32 segments while nothing is
// known about the root (uniform sections), 8 x 64 for the first ladder of a warm start, 4 x 128 afterwards.
//
// One round, for one group of 4 energies and S = 32 SW segments:
//   pre    lanes = energies: far cut-off index, the two far seeds (Numerov.h:294-303) and the real solution down to the next tile boundary
//          q_e (<= 9 nodes): count, product of d, state (W, D) at q_e;
//   main   lane j = tiles [m_lo_j, m_hi_j] of 8 nodes, walked downwards; the per-node tables (a, b12, c6) of the 32 rows of a warp are
//          staged through shared memory with cp.async one tile ahead (row stride 9 doubles: conflict-free).  Every energy pushes the two
//          basis states (W, D) = (1, 0), (0, 1) through the lane's nodes: its 2x2 transfer matrix, the sign changes of the first chain,
//          the product of d_i d_{i+1}.  The coefficient stream (g, s, 10 g) runs from the lane's top for every energy; the chains of an
//          energy whose seeds lie inside the lane are reset to the basis at the first tile below q_e (tile-granular predicate): the loop
//          has no divergent path;
//   scan   inclusive prefix product of the maps over the lanes (5 shuffle steps) and over the sub-warps (shared memory): entry state of
//          every lane = prefix x seed state; the sign changes of the real solution inside a lane follow from the rotation argument of
//          numerov_seg.cu (count of the first basis chain + [end past L] - [start past L]): no second sweep;
//   post   lanes = energies (warp 0): the real solution through nodes 7 .. 1 with the exact formulas (sign of d_1 for l = 3, SURVEY fact
//          6) and y_0 (Numerov.h:398); then the bracket update and the next round's energies.
// Uniform grids (methods 2 / 3: seeds off the nodes) stay on numerov_seg.cu.
#include "numerov_common.cuh"
#include <cstdio>

namespace dft {

constexpr int kRowT = 8;                          // nodes per staged tile
constexpr int kRowE = 4;                          // trial energies per thread
constexpr int kRowWarps = 4;                      // warps per CTA (= per orbital): the throughput shape; kRowWarpsWide = 8: the latency shape (few orbitals left)
constexpr int kRowWarpsWide = 8;
constexpr int kRowMaxW = 8;
constexpr int kRowMaxE = 16;                      // trial energies per round in the widest mode (4 groups of 4)
constexpr int kRowStride = kRowT + 1;             // doubles per staged row (odd: LDS.64 of 32 rows is conflict-free)
constexpr int kRowArr = 32 * kRowStride;          // one table of one stage
constexpr int kRowStage = 3 * kRowArr;            // a, b12, c6
constexpr int rows_smem_bytes(int nw) { return nw * 2 * kRowStage * (int)sizeof(double); }
constexpr int kRowSmemBytes = rows_smem_bytes(kRowWarps);

struct RowShared {
    double E[kRowMaxE];                           // trial energies of the round, ascending
    int n_groups;                                 // NG: energy groups of the round (1, 2 or 4); SW = kRowWarps / NG sub-warps each
    int go;                                       // 1: another round follows
    int use_hint;                                 // 1: the bracket is narrow, the cut-off index of the last round is a good first estimate
    double tot[kRowMaxW][kRowE][4];              // the composed map of a warp's 32 lanes (ww, wd, dw, dd)
    double ptot[kRowMaxW][kRowE];                // product of d over the warp's lanes
    int cnt[kRowMaxW][kRowE];                    // sign changes of the real solution inside the warp's lanes
    int bad[kRowMaxW][kRowE];
    // per energy of the round: what the pre phase found (written by the first sub-warp of the group) and the state entering node 7
    double preP[kRowMaxE], botW[kRowMaxE], botD[kRowMaxE];
    int preCnt[kRowMaxE], preBad[kRowMaxE], start[kRowMaxE];
};

__device__ __forceinline__ void cp_async8(unsigned dst, const double* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ double lds_f64(unsigned addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

struct RowPre {            // pre phase of one energy (lanes = energies)
    int start, qe, count, bad;
    unsigned prev;
    double W, D, P;        // state at node qe: (W_qe, W_qe - W_{qe+1}); P = product of d_i d_{i+1} over the even nodes qe .. start
};

// far cut-off index of the inward sweep = start_index(g, kappa) (numerov_common.cuh; Numerov.h:119-136), warp-collective: lane = 4 j + e
// evaluates the far-value predicate of energy e (= lane & 3, every lane passes its own kappa) at candidate j of a window of 8 indices around
// the closed-form estimate; one evaluation per lane instead of a serial walk.  hint: a cut-off index found earlier for a nearby energy
// (one fixed-point step is then enough), or < 0.  The result is defined by the predicate alone, so it does not depend on the hint.
__device__ __forceinline__ int rows_start(const GridDev& g, double kappa, int hint, int lane)
{
    const unsigned full = 0xffffffffu;
    if (g.uniform) return start_index(g, kappa);
    const int nmax = g.N - 1;
    double x = hint > 0 ? (double)hint : (double)nmax;
    const int iters = hint > 0 ? 1 : 2;
    for (int it = 0; it < iters; ++it) {           // r* kappa + idx delta/2 = 460.5 with r = Rp (e^{delta idx} - 1)
        const double rr = (-kFarLog - x * (0.5 * g.delta)) / kappa;
        x = rr > 0. ? log1p(rr / g.rp) / g.delta : 1.;
        x = fmin(fmax(x, 1.), (double)nmax);
    }
    const int j = lane >> 2;
    const int c = min(max((int)x - 2 + j, 2), nmax);
    const bool below = c >= nmax ? true : far_below(g, kappa, c);
    const unsigned m = (__ballot_sync(full, below) >> (lane & 3)) & 0x11111111u;        // bit 4 j: candidate j of this lane's energy
    const int c0 = min(max((int)x - 2, 2), nmax);
    int res = -1;
    if (m) {
        const int jf = (__ffs((int)m) - 1) >> 2;    // first candidate below the threshold; the one before it (if any) is above
        if (jf > 0 || c0 == 2) res = min(max((int)x - 2 + jf, 2), nmax);
    }
    if (__any_sync(full, res < 0)) { const int r2 = start_index(g, kappa); if (res < 0) res = r2; }      // (estimate off by more than the window)
    return res;
}

__device__ __forceinline__ RowPre rows_pre(const GridDev& g, const double* __restrict__ atab, double ll1, double E, int hint, int lane)
{
    RowPre o;
    const double kappa = sqrt(2. * fabs(E));
    const int start = rows_start(g, kappa, hint, lane);
    o.start = start;
    o.qe = ((start - 1) / kRowT) * kRowT;
    o.bad = o.qe < 2 * kRowT;                      // no main tile below the seeds: the generic serial sweep takes the round
    double W1 = 0., W2 = 0., D = 0., g1 = 0., s1 = 0., t1 = 0., P = 1.;
    unsigned prev = 0;
    int count = 0, bad = 0;
    if (!o.bad) {
        // nodes qe .. qe + kRowT (qe < start <= qe + kRowT) and the two seed nodes again by their own index: one batch of independent loads
        double gv[kRowT + 1];
#pragma unroll
        for (int j = 0; j <= kRowT; ++j) {
            const int i = min(o.qe + j, g.N - 1);
            gv[j] = fma(-E, __ldg(g.c6 + i), fma(ll1, __ldg(g.b12 + i), __ldg(atab + i)));
        }
        const double gs = fma(-E, __ldg(g.c6 + start), fma(ll1, __ldg(g.b12 + start), __ldg(atab + start)));
        const double gt = fma(-E, __ldg(g.c6 + start - 1), fma(ll1, __ldg(g.b12 + start - 1), __ldg(atab + start - 1)));
        const double fs = far_value(g, kappa, start, start), ft = far_value(g, kappa, start - 1, start);
        {   // w_start = d_start far(start), d_{start+1} := 1   (Numerov.h:294-298)
            const double d = 1. - gs;
            W2 = d * fs;
            bad |= !(d > 0.);
            if (!(start & 1)) P *= (1. - gs);
        }
        {   // w_{start-1} d_start   (Numerov.h:300-303)
            const double d = 1. - gt;
            W1 = d * ft * (1. - gs);
            s1 = fma(-gt, gs, gt + gs);
            D = W1 - W2;
            bad |= !(d > 0.);
            if (!((start - 1) & 1)) P *= (1. - s1);
            g1 = gt; t1 = 10. * gt;
        }
        const int js = start - o.qe;               // 1 .. kRowT: the seeds are rows js, js - 1 of the batch
#pragma unroll
        for (int j = kRowT - 2; j >= 0; --j) {
            if (j >= js - 1) continue;
            const double gk = gv[j];
            const double d = 1. - gk;
            const double Dnew = fma(t1, W1, fma(s1, W2, D));
            const double W = W1 + Dnew;
            const double s = fma(-gk, g1, gk + g1);
            const unsigned sy = ((unsigned)hi32(W) ^ (unsigned)hi32(d)) >> 31;
            count += (sy != prev);
            prev = sy;
            bad |= !(d > 0.);
            if (!((o.qe + j) & 1)) P *= (1. - s);
            D = Dnew; W2 = W1; W1 = W; g1 = gk; s1 = s; t1 = 10. * gk;
        }
    }
    o.bad |= bad;
    o.W = W1; o.D = D; o.P = P; o.count = count; o.prev = prev;
    return o;
}

struct RowOut { int cfull, y0_pos, start, bad; double d_first, y0s, P; };      // y_0 = y0s / P (P > 0); its log2: rows_ylog
__device__ __forceinline__ double rows_ylog(double y0s, double P) { return (fabs(y0s) <= 1.7e308) ? log2(fabs(y0s)) - log2(fabs(P)) : INFINITY; }
#ifdef DFT_ROWS_DEBUG
__device__ long long g_rows_clk[12];
__device__ __forceinline__ bool getenv_dbg_clk(unsigned long long* work) { return work != nullptr && (atomicAdd(work + 5, 0ULL) % 50) == 0; }
#define ROWS_CLK(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd((unsigned long long*)&g_rows_clk[i], (unsigned long long)(t_ - t_last)); t_last = t_; } } while (0)
#else
#define ROWS_CLK(i) do { } while (0)
#endif

// post phase of one energy (lanes = energies): the real solution from its state at node kRowT (W_8, W_8 - W_9) through nodes 7 .. 1, y_0
__device__ __forceinline__ RowOut rows_post(const GridDev& g, const double* __restrict__ atab, double ll1, double E, double Win, double Din,
                                            int count_in, double P_in, int bad_in)
{
    const double ga = fma(-E, __ldg(g.c6 + kRowT), fma(ll1, __ldg(g.b12 + kRowT), __ldg(atab + kRowT)));
    const double gb = fma(-E, __ldg(g.c6 + kRowT + 1), fma(ll1, __ldg(g.b12 + kRowT + 1), __ldg(atab + kRowT + 1)));
    double W1 = Win, D = Din, W2 = Win - Din, g1 = ga, s1 = fma(-ga, gb, ga + gb), t1 = 10. * ga, P = P_in;
    unsigned prev = ((unsigned)hi32(W1) ^ (unsigned)hi32(1. - ga)) >> 31;
    int count = count_in, bad = bad_in;
#pragma unroll
    for (int i = kRowT - 1; i >= 1; --i) {
        const double gk = fma(-E, __ldg(g.c6 + i), fma(ll1, __ldg(g.b12 + i), __ldg(atab + i)));
        const double d = 1. - gk;
        const double Dnew = fma(t1, W1, fma(s1, W2, D));
        const double W = W1 + Dnew;
        const double s = fma(-gk, g1, gk + g1);
        const unsigned sy = ((unsigned)hi32(W) ^ (unsigned)hi32(d)) >> 31;      // y_i = W_i / (P_i d_i), P_i > 0
        count += (sy != prev);
        prev = sy;
        if (i == 2) bad |= !(d > 0.);
        if (!(i & 1)) P *= (1. - s);
        D = Dnew; W2 = W1; W1 = W; g1 = gk; s1 = s; t1 = 10. * gk;
    }
    // W1 = W_1, W2 = W_2, g1 = g_1, P = prod_{j=2..start} d_j;  y_0 = y_1 (2 + f_1) - y_2  (Numerov.h:398)
    RowOut o;
    const double d1 = 1. - g1;
    const double Y0s = W1 * fma(12., g1, 2.) / d1 - W2;
    o.y0_pos = Y0s > 0.;
    o.y0s = Y0s; o.P = P;
    o.cfull = count + (((o.y0_pos ? 0u : 1u) != prev) ? 1 : 0);
    o.bad = bad | !(P > 0.);
    o.d_first = d1;
    o.start = 0;
    return o;
}

// One round of n = 4 NG trial energies (sh.E, ascending) by the whole CTA.  On return lane e < n of warp 0 holds the result of energy e
// (other threads: undefined).  Contains block barriers: every thread of the CTA must call it.
__device__ __forceinline__ RowOut rows_round(const GridDev& g, const double* __restrict__ atab, double ll1, int l, int want, RowShared& sh,
                                             unsigned tiles_smem, int warp, int lane, int n_warps = kRowWarps, int* hint_io = nullptr)
{
    const unsigned full = 0xffffffffu;
    const int NG = sh.n_groups, SW = n_warps / NG;
    const int gi = warp / SW, si = warp - gi * SW;
    const int S = 32 * SW;
    const int nmax = g.N - 1;

#ifdef DFT_ROWS_DEBUG
    long long t_last = clock64();
#endif
    // ---------------- pre: seeds (lane = energy lane & 3 of the group, replicated over the warp) ----------------
    const int eg = gi * kRowE + (lane & 3);
    const RowPre pre = rows_pre(g, atab, ll1, sh.E[eg], hint_io ? *hint_io : -1, lane);
    if (hint_io) *hint_io = pre.start;
    if (si == 0 && lane < kRowE) { sh.preP[eg] = pre.P; sh.preCnt[eg] = pre.count; sh.preBad[eg] = pre.bad; sh.start[eg] = pre.start; }
    double E[kRowE], seedW[kRowE], seedD[kRowE];
    int mf[kRowE];                                 // first (highest) main tile of the energy
    int M = 1;
#pragma unroll
    for (int e = 0; e < kRowE; ++e) {
        E[e] = sh.E[gi * kRowE + e];
        seedW[e] = __shfl_sync(full, pre.W, e);
        seedD[e] = __shfl_sync(full, pre.D, e);
        mf[e] = __shfl_sync(full, pre.qe, e) / kRowT - 1;
        M = max(M, mf[e]);
    }
    // ---------------- segmentation: tiles 1 .. M dealt from the bottom, tpl tiles per lane ----------------
    const int tpl = (M + S - 1) / S;
    const int S_used = (M + tpl - 1) / tpl;
    const int j = si * 32 + lane;                  // 0 = top
    const bool valid = j < S_used;
    const int m_lo = 1 + (S_used - 1 - j) * tpl;   // (negative for the lanes below the bottom: masked)
    const int m_hi = m_lo + tpl - 1;
    const int tile_cap = nmax / kRowT - 1;         // highest tile that is read whole
    int kfirst[kRowE];
    bool active[kRowE];
#pragma unroll
    for (int e = 0; e < kRowE; ++e) {
        kfirst[e] = max(0, m_hi - mf[e]);
        active[e] = valid && mf[e] >= 1 && kfirst[e] <= tpl - 1;
    }
    // staging: this warp's two stages; row = lane of this warp
    const unsigned stage0 = tiles_smem + (unsigned)(warp * 2 * kRowStage * sizeof(double));
    const int row_j0 = S_used - 1 - si * 32;        // row r of this warp is segment (from the bottom) row_j0 - r
    auto prefetch = [&](int step, int buf) {
        const unsigned sb = stage0 + (unsigned)(buf * kRowStage * sizeof(double));
#pragma unroll
        for (int q = 0; q < kRowT; ++q) {
            const int idx = lane + 32 * q;
            const int row = idx >> 3, col = idx & 7;
            int tile = 1 + (row_j0 - row) * tpl + tpl - 1 - step;
            tile = min(max(tile, 0), tile_cap);
            const int node = tile * kRowT + col;
            const unsigned dst = sb + (unsigned)((row * kRowStride + col) * sizeof(double));
            cp_async8(dst, atab + node);
            cp_async8(dst + (unsigned)(kRowArr * sizeof(double)), g.b12 + node);
            cp_async8(dst + (unsigned)(2 * kRowArr * sizeof(double)), g.c6 + node);
        }
        cp_async_commit();
    };
    ROWS_CLK(0);
    prefetch(0, 0);

    // coefficient carries at the lane's top: g_{top+1}, s_{top+1} = 1 - d_{top+1} d_{top+2}, 10 g_{top+1}
    double g1[kRowE], s1[kRowE], t1[kRowE];
    {
        const int i1 = min(max((m_hi + 1) * kRowT, 0), nmax), i2 = min(max((m_hi + 1) * kRowT + 1, 0), nmax);
        const double a1 = __ldg(atab + i1), b1 = __ldg(g.b12 + i1), c1 = __ldg(g.c6 + i1);
        const double a2 = __ldg(atab + i2), b2 = __ldg(g.b12 + i2), c2 = __ldg(g.c6 + i2);
        const double g01 = fma(ll1, b1, a1), g02 = fma(ll1, b2, a2);
#pragma unroll
        for (int e = 0; e < kRowE; ++e) {
            const double ga = fma(-E[e], c1, g01), gb = fma(-E[e], c2, g02);
            g1[e] = ga; s1[e] = fma(-ga, gb, ga + gb); t1[e] = 10. * ga;
        }
    }
    // chains: u enters as (W, D) = (1, 0), v as (0, 1);  W2 = W_{i+2} = W - D
    double Wu1[kRowE], Wu2[kRowE], Du[kRowE], Wv1[kRowE], Wv2[kRowE], Dv[kRowE], P[kRowE];
    unsigned sb[kRowE];
    int count[kRowE], gmax[kRowE];
#pragma unroll
    for (int e = 0; e < kRowE; ++e) {
        Wu1[e] = 1.; Wu2[e] = 1.; Du[e] = 0.; Wv1[e] = 0.; Wv2[e] = -1.; Dv[e] = 1.; P[e] = 1.;
        sb[e] = 0; count[e] = 0; gmax[e] = 0;
    }
    ROWS_CLK(1);
    // ---------------- main loop ----------------
    for (int k = 0; k < tpl; ++k) {
        cp_async_wait_all();
        __syncwarp();
        if (k + 1 < tpl) prefetch(k + 1, (k + 1) & 1);
        const unsigned tb = stage0 + (unsigned)(((k & 1) * kRowStage + lane * kRowStride) * sizeof(double));
#pragma unroll
        for (int e = 0; e < kRowE; ++e) {
            if (k == kfirst[e]) {                  // the first tile below this energy's seeds (or the lane's top): enter with the basis
                Wu1[e] = 1.; Wu2[e] = 1.; Du[e] = 0.; Wv1[e] = 0.; Wv2[e] = -1.; Dv[e] = 1.; P[e] = 1.;
                sb[e] = 0; count[e] = 0; gmax[e] = 0;
            }
        }
#pragma unroll
        for (int c = kRowT - 1; c >= 0; --c) {
            const double av = lds_f64(tb + (unsigned)(c * sizeof(double)));
            const double bv = lds_f64(tb + (unsigned)((kRowArr + c) * sizeof(double)));
            const double cv = lds_f64(tb + (unsigned)((2 * kRowArr + c) * sizeof(double)));
            const double g0 = fma(ll1, bv, av);
#pragma unroll
            for (int e = 0; e < kRowE; ++e) {
                const double gk = fma(-E[e], cv, g0);
                const double sn = fma(-gk, g1[e], gk + g1[e]);
                const double Dun = fma(t1[e], Wu1[e], fma(s1[e], Wu2[e], Du[e]));
                const double Dvn = fma(t1[e], Wv1[e], fma(s1[e], Wv2[e], Dv[e]));
                const double Wu = Wu1[e] + Dun, Wv = Wv1[e] + Dvn;
                sb[e] = __funnelshift_l((unsigned)hi32(Wu), sb[e], 1);
                gmax[e] = max(gmax[e], hi32(gk));
                if (!(c & 1)) P[e] *= (1. - sn);   // tiles start at even nodes: even column <=> even node
                Wu2[e] = Wu1[e]; Wu1[e] = Wu; Du[e] = Dun;
                Wv2[e] = Wv1[e]; Wv1[e] = Wv; Dv[e] = Dvn;
                g1[e] = gk; s1[e] = sn; t1[e] = 10. * gk;
            }
        }
#pragma unroll
        for (int e = 0; e < kRowE; ++e) count[e] += __popc((sb[e] ^ (sb[e] >> 1)) & 0xffu);     // bit 8 = sign at the node above the tile
    }

    ROWS_CLK(2);
    // ---------------- scan of the maps over the lanes ----------------
    double ia[kRowE], ib[kRowE], ic[kRowE], id[kRowE];      // inclusive prefix (ww, wd, dw, dd)
#pragma unroll
    for (int e = 0; e < kRowE; ++e) {
        ia[e] = active[e] ? Wu1[e] : 1.; ib[e] = active[e] ? Wv1[e] : 0.;
        ic[e] = active[e] ? Du[e] : 0.;  id[e] = active[e] ? Dv[e] : 1.;
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
        for (int e = 0; e < kRowE; ++e) {
            const double ja = __shfl_up_sync(full, ia[e], o), jb = __shfl_up_sync(full, ib[e], o);
            const double jc = __shfl_up_sync(full, ic[e], o), jd = __shfl_up_sync(full, id[e], o);
            if (lane >= o) {                        // this map after the maps above it
                const double na = fma(ia[e], ja, ib[e] * jc), nb = fma(ia[e], jb, ib[e] * jd);
                const double nc = fma(ic[e], ja, id[e] * jc), nd = fma(ic[e], jb, id[e] * jd);
                ia[e] = na; ib[e] = nb; ic[e] = nc; id[e] = nd;
            }
        }
    }
    if (lane == 31) {
#pragma unroll
        for (int e = 0; e < kRowE; ++e) { sh.tot[warp][e][0] = ia[e]; sh.tot[warp][e][1] = ib[e]; sh.tot[warp][e][2] = ic[e]; sh.tot[warp][e][3] = id[e]; }
    }
    __syncthreads();
    int lane_bad = 0;
#pragma unroll
    for (int e = 0; e < kRowE; ++e) {
        // state entering this warp's top lane: the sub-warps above, applied to the seed state
        double A = seedW[e], B = seedD[e];
        for (int v = 0; v < si; ++v) {
            const double* t = sh.tot[gi * SW + v][e];
            const double na = fma(t[0], A, t[1] * B), nb = fma(t[2], A, t[3] * B);
            A = na; B = nb;
        }
        if (si == SW - 1 && lane == 31) {           // the state entering node 7: everything applied
            sh.botW[gi * kRowE + e] = fma(ia[e], A, ib[e] * B);
            sh.botD[gi * kRowE + e] = fma(ic[e], A, id[e] * B);
        }
        // exclusive prefix of this lane
        double xa = __shfl_up_sync(full, ia[e], 1), xb = __shfl_up_sync(full, ib[e], 1);
        double xc = __shfl_up_sync(full, ic[e], 1), xd = __shfl_up_sync(full, id[e], 1);
        if (lane == 0) { xa = 1.; xb = 0.; xc = 0.; xd = 1.; }
        const double Aj = fma(xa, A, xb * B), Bj = fma(xc, A, xd * B);
        // sign changes of the real solution W = A u + B v inside the lane (numerov_seg.cu: rotation argument)
        const double ue = Wu1[e], ve = Wv1[e];
        const double We = fma(Aj, ue, Bj * ve);
        const double sl = Bj < 0. ? -1. : (Bj > 0. ? 1. : (Aj >= 0. ? 1. : -1.));
        const int past0 = (sl * Aj >= 0.) ? 1 : 0;
        const int past1 = ((ue >= 0. ? 1. : -1.) * sl * We >= 0.) ? 1 : 0;
        int cnt = active[e] ? count[e] + past1 - past0 : 0;
        double pj = active[e] ? P[e] : 1.;
        int bj = active[e] ? ((gmax[e] >= 0x3ff00000) | !(P[e] > 0.)) : 0;       // some 1 - f/12 <= 0 inside the lane
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            cnt += __shfl_xor_sync(full, cnt, o);
            pj *= __shfl_xor_sync(full, pj, o);
            bj |= __shfl_xor_sync(full, bj, o);
        }
        if (lane == 0) { sh.cnt[warp][e] = cnt; sh.ptot[warp][e] = pj; sh.bad[warp][e] = bj; }
        lane_bad |= bj;
    }
    __syncthreads();

    ROWS_CLK(3);
    // ---------------- post: nodes 7 .. 1 and y_0, lane = energy (warp 0) ----------------
    RowOut r;
    r.cfull = 0; r.y0_pos = 0; r.start = 0; r.bad = 0; r.d_first = 1.; r.y0s = 1.; r.P = 1.;
    if (warp == 0) {
        const int n = NG * kRowE;
        const int e = min(lane, n - 1);
        const int ge = e / kRowE, qe = e - ge * kRowE;
        int cnt = sh.preCnt[e], bad = sh.preBad[e];
        double Pt = sh.preP[e];
        for (int v = 0; v < SW; ++v) { cnt += sh.cnt[ge * SW + v][qe]; Pt *= sh.ptot[ge * SW + v][qe]; bad |= sh.bad[ge * SW + v][qe]; }
        r = rows_post(g, atab, ll1, sh.E[e], sh.botW[e], sh.botD[e], cnt, Pt, bad);
        r.start = sh.start[e];
        if (__any_sync(full, r.bad)) {
            // a non-positive 1 - f/12 inside the sweep, or a sweep too short to cut (grid far too coarse for this energy): generic serial path
            const LaneOut so = sweep_lane(g, atab, l, sh.E[e], want);
            r.cfull = so.count_full; r.d_first = so.d_first; r.y0_pos = so.y0_pos; r.P = 1.;
            r.y0s = (so.y0_log2 > -1e300 && so.y0_log2 < 1e300) ? (so.y0_pos ? 1. : -1.) * exp2(fmin(fmax(so.y0_log2, -1000.), 1000.)) : INFINITY;
        }
    }
#ifdef DFT_ROWS_DEBUG
    if (r.y0s == 1.2345e-300 && r.P == 7. && r.cfull == 12345) sh.go = 2;       // (the clock below must wait for the results)
#endif
    ROWS_CLK(4);
    return r;
}

// ---------------------------------------------------------------------------------------------------------
// bracket of one level with n <= 16 samples per round (lanes 0 .. n-1 of warp 0); the 32-sample version is numerov_common.cuh: Bracket.
// The predicate is monotone, so every ascending sample set brackets the same root; the shapes only decide how fast:
//   kSection : n points that cut [lo, hi] into n + 1 equal parts (nothing is known, or y0 is still far from linear over the bracket);
//   kLadder  : c -+ inner g^m (m = 0 .. n/2 - 1, outermost offset = radius) around an estimate c of the root;
//   kOneSide : after a round whose samples all fell on one side of the root: anchor +- d0 g^m from the last sample towards the bracket end
//              (the miss says nothing about the distance: every scale between the ladder's span and the bracket gets a point).
// ---------------------------------------------------------------------------------------------------------
enum { kSection = 0, kLadder = 1, kOneSide = 2 };
struct RowBracket {
    double lo, hi;          // the root is in (lo, hi]
    double c_est, radius;   // kLadder: centre and outermost offset;  kOneSide: anchor and first offset
    double inner;           // kLadder: innermost offset
    double y_lm, P_lm;      // y_0 = y_lm / P_lm of the last virtual-bisection midpoint (1e15 guard, DFTAtom.cpp:528)
    int mode;
    int side;               // kOneSide: -1 = the root lies below the anchor, +1 = above
    bool trusted;           // kLadder: the estimate comes from a checked interpolation (4 energies are enough for the round)
};

__device__ __forceinline__ double rows_sample(const RowBracket& b, int e, int n)
{
    if (b.mode == kLadder) {
        const int h = n >> 1;
        const double inner = fmin(b.inner, b.radius);
        const int mstep = (e < h) ? (h - 1 - e) : (e - h);                  // 0 = closest to the estimate
        double off;
        if (h == 2) off = mstep ? fmax(b.radius, inner) : inner;            // (the production shape: 4 energies per round)
        else {
            const double lg = h > 1 ? log2(fmax(b.radius, inner) / inner) / (double)(h - 1) : 0.;
            off = inner * exp2((double)mstep * lg);
        }
        return fmin(fmax((e < h) ? b.c_est - off : b.c_est + off, b.lo), b.hi);
    }
    if (b.mode == kOneSide) {
        const double far = b.side < 0 ? b.c_est - b.lo : b.hi - b.c_est;
        const double d0 = fmin(b.radius, far);
        const int mstep = b.side < 0 ? (n - 1 - e) : e;
        double off;
        if (n == 4) {                                                       // ratio^(mstep / 4) from two square roots
            const double q = sqrt(sqrt(fmax(far / d0, 1.)));
            off = d0 * (mstep & 1 ? q : 1.) * (mstep & 2 ? q * q : 1.);
        } else {
            const double lg = log2(fmax(far / d0, 1.)) / (double)n;         // the n-th step would land on the bracket end
            off = d0 * exp2((double)mstep * lg);
        }
        return fmin(fmax(b.side < 0 ? b.c_est - off : b.c_est + off, b.lo), b.hi);
    }
    return b.lo + (b.hi - b.lo) * ((double)(e + 1) / (double)(n + 1));
}

// warp-collective (warp 0): lanes >= n pass copies of lane n-1; all lanes end with the same bracket
__device__ __forceinline__ void rows_update(RowBracket& b, int n, double E, bool high, double y0s, double P)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned m_hi = __ballot_sync(full, high);
    int lo_i, hi_i, lm;
    virtual_bisect(m_hi, n, lo_i, hi_i, lm);
    const double E_first = __shfl_sync(full, E, 0), E_second = __shfl_sync(full, E, 1);
    const double E_last = __shfl_sync(full, E, n - 1), E_prev = __shfl_sync(full, E, n - 2);
    const double a_lo = __shfl_sync(full, E, max(lo_i, 0)), a_hi = __shfl_sync(full, E, min(hi_i, n - 1));
    const double e_lo = lo_i >= 0 ? a_lo : b.lo, e_hi = hi_i < n ? a_hi : b.hi;
    b.y_lm = __shfl_sync(full, y0s, lm); b.P_lm = __shfl_sync(full, P, lm);
    b.mode = kSection; b.trusted = false;
    // every sample on one side of the root: one-sided ladder towards the bracket end - unless that end is closer than the samples' own span
    // (it is then a sample of an earlier round: equal sections of what is left)
    if (lo_i < 0 && hi_i < n && E_first - b.lo > 2. * (E_last - E_first)) {
        b.mode = kOneSide; b.side = -1; b.c_est = E_first; b.radius = fmax(E_second - E_first, 16. * kLadderEps);
    } else if (hi_i == n && lo_i >= 0 && b.hi - E_last > 2. * (E_last - E_first)) {
        b.mode = kOneSide; b.side = 1; b.c_est = E_last; b.radius = fmax(E_last - E_prev, 16. * kLadderEps);
    }
    // estimate of the root for the next round: zero of y0(E) through the samples around the sign change.  The outer two of the four
    // must be WELL SEPARATED from the bracketing pair (>= 5 % of its width): after a round whose innermost pair (+-0.45 energyErr) missed
    // the root, that pair is 1e-12 apart and its divided difference is rounding noise
    if (lo_i >= 0 && hi_i < n && e_lo < e_hi) {
        double Ek[4], yk[4], Pk[4];
        bool ok[4];
        double ref = 0.;
        const double thr = 0.05 * (e_hi - e_lo);
        const unsigned mL = __ballot_sync(full, lane < lo_i && (e_lo - E) >= thr);
        const unsigned mR = __ballot_sync(full, lane > hi_i && lane < n && (E - e_hi) >= thr);
        const int pick[4] = { mL ? 31 - __clz((int)mL) : -1, lo_i, hi_i, mR ? __ffs((int)mR) - 1 : -1 };
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int idx = pick[q];
            const int src_lane = min(max(idx, 0), n - 1);
            Ek[q] = __shfl_sync(full, E, src_lane);
            yk[q] = __shfl_sync(full, y0s, src_lane);
            Pk[q] = __shfl_sync(full, P, src_lane);
            ok[q] = idx >= 0 && idx < n && fabs(yk[q]) <= 1.7e308 && yk[q] != 0. && Pk[q] > 0.;
            if (ok[q]) ref = fmax(ref, fabs(yk[q]));
        }
        // y_0 = y0s / P of the usable samples up to one common positive factor (no division, no logarithm): y0s relative to the largest
        // one, times the P of the OTHER usable samples
        const double inv = 1. / ref;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            double v = ok[q] ? yk[q] * inv : 0.;
#pragma unroll
            for (int r = 0; r < 4; ++r) if (r != q && ok[r]) v *= Pk[r];
            yk[q] = v;
        }
        // the bracket ends must be proper samples with opposite signs and distinct energies
        if (ok[1] && ok[2] && yk[1] * yk[2] < 0. && Ek[1] < Ek[2]) {
            const double dE = Ek[2] - Ek[1], dy = yk[2] - yk[1];
            const double E2 = Ek[1] - yk[1] * (dE / dy);                                  // secant
            // An outer point is usable when it extends the table monotonically in E and in y (inverse interpolation) AND the line through
            // the bracketing pair predicts it within a factor 4: y0(E) = (E - E*) x (a factor that varies exponentially with E) - over a
            // bracket that is still wide the pair's smaller value is ~0 next to the larger one, every interpolant passes through that end
            // and agrees with every other one: agreement between secant and cubic alone proves nothing
            bool lin[4];
#pragma unroll
            for (int q = 0; q < 4; q += 3) {
                const double pd = fma(Ek[q] - Ek[1], dy, yk[1] * dE);                     // (the line's prediction) x dE, dE > 0
                const double yd = yk[q] * dE;
                lin[q] = (pd > 0.) == (yd > 0.) && fabs(yd) > 0.25 * fabs(pd) && fabs(yd) < 4. * fabs(pd);
            }
            const bool use0 = ok[0] && Ek[0] < Ek[1] && (yk[0] - yk[1]) * (yk[1] - yk[2]) > 0. && lin[0];
            const bool use3 = ok[3] && Ek[3] > Ek[2] && (yk[2] - yk[3]) * (yk[1] - yk[2]) > 0. && lin[3];
            double Eh = E2;
            if (use0 || use3) {                                                           // inverse Lagrange interpolation at y = 0: one division per point
                double num = 0.;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const bool uq = (q == 0) ? use0 : (q == 3 ? use3 : true);
                    if (!uq) continue;
                    double top = Ek[q], bot = 1.;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const bool ur = (r == 0) ? use0 : (r == 3 ? use3 : true);
                        if (r == q || !ur) continue;
                        top *= -yk[r]; bot *= yk[q] - yk[r];
                    }
                    num += top / bot;
                }
                Eh = num;
            }
            if ((use0 || use3) && Eh > e_lo && Eh < e_hi) {
                b.c_est = Eh;
                b.radius = fmin(fmax(4. * fabs(Eh - E2), 16. * kLadderEps), fmax(e_hi - Eh, Eh - e_lo));
                // innermost pair: +-0.45 energyErr (the bracket closes in this round when the estimate is that good)
                b.inner = 0.45 * kEnergyTol;
                b.mode = kLadder; b.trusted = true;
            }
            // (no checked third point: the next round cuts [e_lo, e_hi] into equal parts - a factor n + 1 whatever y0 looks like)
        }
    }
    b.lo = e_lo; b.hi = e_hi;
}

// cfg: energy groups per round (1, 2 or 4) for [bits 0-3] the first ladder of a warm start, [4-7] later ladders, [8-11] uniform rounds
template <int NW>
__global__ void __launch_bounds__(32 * NW, NW == kRowWarps ? 3 : 1) search_rows_kernel(GridDev g, const double* __restrict__ atab_all, const AtomDev* atoms,
                                                                      const OrbitalDev* orbs, const AtomState* astate, SearchState* ss, int n_orbs,
                                                                      unsigned long long* work, int warm_start, int cfg, int step_min, int step_max)
{
    DFT_PDL_WAIT();
    extern __shared__ __align__(16) unsigned char rows_smem[];
    __shared__ RowShared sh;
#ifdef DFT_ROWS_DEBUG
    long long t_mark = clock64();
#endif
    const unsigned full = 0xffffffffu;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = blockIdx.x;
    if (k >= n_orbs) return;
    const OrbitalDev ob = orbs[k];
    if (astate[ob.atom].done) return;
    { const int sc = astate[ob.atom].n_steps; if (sc < step_min || sc >= step_max) return; }      // (the two shapes of the kernel share an SCF by step index)
    const double* __restrict__ atab = atab_all + (size_t)ob.tab * g.N;
    const double ll1 = (double)(ob.l * (ob.l + 1));
    const double Z = (double)atoms[ob.atom].Z;
    const unsigned tiles_smem = (unsigned)__cvta_generic_to_shared(rows_smem);
    RowBracket b;
    b.lo = -Z * Z - 1.; b.hi = kTopEnergy;                // DFTAtom.cpp:407,499
    b.y_lm = 1.; b.P_lm = 1.; b.side = 0; b.trusted = false;
    const SearchState s0 = ss[k];
    const bool warm = (warm_start & 1) && s0.pad == 1;
    b.mode = warm ? kLadder : kSection;
    // first ladder: the levels move geometrically from one SCF step to the next (linear mixing); centre = previous eigenvalue + last
    // shift x (ratio of the last two shifts), radius = 1.5 x last shift, innermost offset = twice what the last step's prediction missed by
    const double e_prev = s0.E, sh1 = s0.up_lo, sh2 = s0.up_hi;
    const double ratio = (sh2 != 0. && fabs(sh1) < fabs(sh2)) ? sh1 / sh2 : 0.;
    b.c_est = fmin(fmax(e_prev + sh1 * ratio, b.lo), b.hi);
    b.radius = fmin(fmax(1.5 * fabs(sh1), 1e-7), Z * Z + 51.);
    b.inner = (s0.dn_lo > 0.) ? fmin(fmax(2. * s0.dn_lo, 0.45 * kEnergyTol), 0.25 * b.radius) : 0.125 * b.radius;
    if (warm_start & 2) {
        // Inside an SCF (the step counter of the atom says where): what the first steps of the reference's SCF are known to do.  Only the
        // first ladder changes - a wrong guess costs rounds, never the result (the bracket logic certifies every bracket it keeps).
        const int sc = astate[ob.atom].n_steps;
        const double mix = atoms[ob.atom].mixing;
        if (sc == 0 && !warm) {
            // step 0: the initial density is a uniform sphere of Q electrons and radius MaxR (DFTAtom.cpp:371-376): V = -Z/r + 3Q/(2 MaxR)
            // - Q r^2/(2 MaxR^3) + v_xc of a density of ~1e-3: hydrogenic levels shifted by 3Q/(2 MaxR) - ~0.1
            const double nq = (double)(ob.want + ob.l + 1);
            const double hyd = Z * Z / (2. * nq * nq);
            const double Q = atoms[ob.atom].n_el[0] + atoms[ob.atom].n_el[1];
            b.mode = kLadder;
            b.c_est = fmin(fmax(-hyd + 1.5 * Q / g.max_r - 0.1, b.lo), b.hi);
            b.inner = 0.1; b.radius = 0.4 + 0.002 * hyd;
        } else if (warm && sc == 1) {
            // step 1: the first real density screens the nucleus: every level rises by about (1 - mixing) x (|E| + 2); samples on that side only
            const double up = 2. * (1. - mix) * sh1;           // (sh1 = 0.5 |E| + 1 after a cold search)
            b.c_est = fmin(fmax(e_prev + 1.025 * up, b.lo), b.hi);
            b.inner = 0.125 * up; b.radius = 0.5 * up;
            if (!(up > 1e-7)) { b.c_est = e_prev; b.inner = 0.125 * b.radius; }
        } else if (warm && sc >= 2) {
            // step 2: one real shift so far - the shifts of a linearly mixed SCF decay by ~1 - 1.28 (1 - mixing) per step (0.36 at mixing 0.5);
            // later: the miss of the extrapolation scales with the shifts
            const bool real2 = sc >= 3;
            const double q = real2 ? ratio : fmax(0., 1. - 1.28 * (1. - mix));
            b.c_est = fmin(fmax(e_prev + sh1 * q, b.lo), b.hi);
            b.radius = fmin(fmax(0.75 * fabs(sh1), 1e-7), Z * Z + 51.);
            const double decay = (real2 && sh2 != 0.) ? fmin(fabs(sh1 / sh2), 1.) : 1.;
            b.inner = real2 ? ((s0.dn_lo > 0.) ? fmin(fmax(2. * s0.dn_lo * decay, 0.45 * kEnergyTol), 0.25 * b.radius) : 0.125 * b.radius)
                            : 0.16 * b.radius;
        }
    }
    const double c_first = b.c_est;
    long long steps = 0;
    int rounds = 0, sweeps = 0, hint = -1;

#ifdef DFT_ROWS_DEBUG
    __shared__ double dbg_hist[16][8];
    const long long t_kernel0 = clock64();
#endif
#ifdef DFT_ROWS_DEBUG
#define ROWS_KCLK(i) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd((unsigned long long*)&g_rows_clk[i], (unsigned long long)(t_ - t_mark)); t_mark = t_; } } while (0)
#else
#define ROWS_KCLK(i) do { } while (0)
#endif
    ROWS_KCLK(10);                                      // prologue
    for (int round = 0; round < 96; ++round) {
        if (warp == 0) {
            const bool go = bracket_open(b.lo, b.hi);
#ifdef DFT_ROWS_DEBUG
            if (lane == 0 && round < 16) {
                dbg_hist[round][0] = b.lo; dbg_hist[round][1] = b.hi; dbg_hist[round][2] = b.c_est; dbg_hist[round][3] = b.radius;
                dbg_hist[round][4] = b.inner; dbg_hist[round][5] = (double)(b.mode * 10 + (b.mode == kOneSide ? b.side + 1 : (int)b.trusted)); dbg_hist[round][6] = 0.;
            }
#endif
            const int NG = b.mode != kLadder ? ((cfg >> 8) & 15) : (b.trusted ? ((cfg >> 4) & 15) : (cfg & 15));      // (NG divides NW: 1, 2 or 4)
            if (lane == 0) { sh.go = go; sh.n_groups = NG; sh.use_hint = round > 0 && (b.hi - b.lo) < 0.02 * fabs(b.lo); }
            const int n = NG * kRowE;
            if (lane < n) sh.E[lane] = rows_sample(b, lane, n);
        }
        __syncthreads();
        if (!sh.go) break;
        const int n = sh.n_groups * kRowE;
        if (!sh.use_hint) hint = -1;
        ROWS_KCLK(9);                                   // sample + barrier
        const RowOut r = rows_round(g, atab, ll1, ob.l, ob.want, sh, tiles_smem, warp, lane, NW, &hint);
        ++rounds; sweeps += n;
#ifdef DFT_ROWS_DEBUG
        if (threadIdx.x == 0) t_mark = clock64();
#endif
        if (warp == 0) {
            const double E = sh.E[min(lane, n - 1)];
            if (lane < n) steps += r.start - 1;
            rows_update(b, n, E, r.cfull > ob.want + (r.d_first < 0. ? 1 : 0), r.y0s, r.P);
        }
#ifdef DFT_ROWS_DEBUG
        if (b.c_est == 1.2345e-300 && b.lo == 7. && b.hi == 8. && b.radius == 9.) sh.go = 2;
#endif
        ROWS_KCLK(8);                                   // bracket update
        __syncthreads();                               // sh.E / sh.go are rewritten at the top
#ifdef DFT_ROWS_DEBUG
        if (threadIdx.x == 0) t_mark = clock64();
#endif
    }
#ifdef DFT_ROWS_DEBUG
    if (threadIdx.x == 0) { atomicAdd((unsigned long long*)&g_rows_clk[5], (unsigned long long)(clock64() - t_kernel0)); atomicAdd((unsigned long long*)&g_rows_clk[6], (unsigned long long)rounds); atomicAdd((unsigned long long*)&g_rows_clk[7], 1ULL); }
    if (threadIdx.x == 0 && k == 0 && getenv_dbg_clk(work)) printf("rows clk: pre %lld prefetch+carry %lld main %lld scan %lld post %lld | update %lld sample+barrier %lld prologue %lld | loop total %lld rounds %lld solves %lld (sum over CTAs so far)\n", g_rows_clk[0], g_rows_clk[1], g_rows_clk[2], g_rows_clk[3], g_rows_clk[4], g_rows_clk[8], g_rows_clk[9], g_rows_clk[10], g_rows_clk[5], g_rows_clk[6], g_rows_clk[7]);
    if (warp == 0 && lane == 0 && rounds >= 6 && s0.pad == 1 && work && atomicAdd(work + 5, 1ULL) % 97 == 0) {
        printf("orb %d l %d want %d e_prev %.12g shifts %.3e %.3e miss_prev %.3e -> E %.12g in %d rounds\n", k, ob.l, ob.want, e_prev, sh1, sh2, s0.dn_lo, b.lo, rounds);
        for (int r = 0; r < min(rounds, 16); ++r)
            printf("   r%d: lo-E %.3e hi-E %.3e c-E %.3e R %.3e inner %.3e kind %g win %.3e\n", r, dbg_hist[r][0] - b.lo, dbg_hist[r][1] - b.lo, dbg_hist[r][2] - b.lo,
                   dbg_hist[r][3], dbg_hist[r][4], dbg_hist[r][5], dbg_hist[r][6]);
    }
#endif
    if (warp == 0) {
        if (lane == 0) {
            SearchState s = s0;
            s.bot = b.lo; s.top = b.hi; s.E = b.lo;                              // level.E = BottomEnergy, DFTAtom.cpp:534
            const double ylog = rows_ylog(b.y_lm, b.P_lm);
            s.y0_log2 = ylog;
            s.converged = (b.hi - b.lo < kEnergyTol) && (ylog < 49.828921423310435);   // DFTAtom.cpp:528
            s.stage = 3;
            s.up_hi = warm ? s0.up_lo : 0.;                                      // the last two shifts of the level
            s.up_lo = warm ? b.lo - e_prev : 0.5 * fabs(b.lo) + 1.;                // (no shift yet: the scale the level may move by)
            s.dn_lo = warm ? fabs(b.lo - c_first) : 0.;                          // what this step's prediction missed by
            s.pad = 1;
            ss[k] = s;
        }
        if (work) {
#pragma unroll
            for (int o = 16; o; o >>= 1) steps += __shfl_xor_sync(full, steps, o);
            if (lane == 0) {
                atomicAdd(work, (unsigned long long)steps);
                atomicAdd(work + DFTATOM_K_MATCH, 1ULL);                          // orbital solves
                atomicAdd(work + DFTATOM_K_DENSITY, (unsigned long long)rounds);  // search rounds
                atomicAdd(work + 7, (unsigned long long)sweeps);                  // inward sweeps (trial energies)
                atomicAdd(work + 8 + min(rounds, 15), 1ULL);                      // histogram (debug aid)
                atomicAdd(work + 24 + min(ob.l, 3), (unsigned long long)rounds);
                if (rounds >= 4) atomicAdd(work + 28 + min(ob.l, 3), 1ULL);
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------
// lanes kernel (component entry point / C5b microbench): one CTA per n = 4 NG consecutive lanes.  Lanes that share (tab, l) go through one
// round together; otherwise the CTA runs one round per lane (all energy slots = that lane), which is what the parity test exercises
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * kRowWarps, 3) numerov_lanes_rows_kernel(GridDev g, NumerovLaneArgs a, int NG)
{
    extern __shared__ __align__(16) unsigned char rows_smem[];
    __shared__ RowShared sh;
    __shared__ int s_same;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = NG * kRowE;
    const int k0 = blockIdx.x * n;
    if (k0 >= a.n_lanes) return;
    const unsigned tiles_smem = (unsigned)__cvta_generic_to_shared(rows_smem);
    if (threadIdx.x == 0) {
        int same = 1;
        for (int q = 1; q < n; ++q) {
            const int kq = min(k0 + q, a.n_lanes - 1);
            same &= (a.tab[kq] == a.tab[k0]) && (a.l[kq] == a.l[k0]);
        }
        s_same = same;
        sh.n_groups = NG;
    }
    __syncthreads();
    const int passes = s_same ? 1 : n;
    for (int p = 0; p < passes; ++p) {
        if (threadIdx.x < n) sh.E[threadIdx.x] = a.E[min(k0 + (s_same ? (int)threadIdx.x : p), a.n_lanes - 1)];
        __syncthreads();
        const int kp = min(k0 + p, a.n_lanes - 1);
        const int l = a.l[kp];
        const RowOut r = rows_round(g, a.atab + (size_t)a.tab[kp] * g.N, (double)(l * (l + 1)), l, a.limit ? a.limit[kp] : 0, sh, tiles_smem, warp, lane);
        if (warp == 0) {
            const int k = s_same ? k0 + lane : k0 + p;
            const bool mine = s_same ? (lane < n) : (lane == 0);
            if (mine && k < a.n_lanes) {
                if (a.y0_sign) a.y0_sign[k] = r.y0_pos;
                if (a.y0_log2) a.y0_log2[k] = rows_ylog(r.y0s, r.P);
                if (a.count) a.count[k] = r.cfull;
            }
        }
        __syncthreads();
    }
}

void launch_numerov_lanes_rows(const GridDev& g, const NumerovLaneArgs& a, int n_groups, cudaStream_t st)
{
    const int NG = (n_groups == 1 || n_groups == 2) ? n_groups : 4;
    const int n = NG * kRowE;
    numerov_lanes_rows_kernel<<<(a.n_lanes + n - 1) / n, 32 * kRowWarps, kRowSmemBytes, st>>>(g, a, NG);
}

int rows_init_device()
{
    cudaError_t e = cudaFuncSetAttribute(search_rows_kernel<kRowWarps>, cudaFuncAttributeMaxDynamicSharedMemorySize, rows_smem_bytes(kRowWarps));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(search_rows_kernel<kRowWarpsWide>, cudaFuncAttributeMaxDynamicSharedMemorySize, rows_smem_bytes(kRowWarpsWide));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(numerov_lanes_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRowSmemBytes);
    if (e != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute(search_rows_kernel): ") + cudaGetErrorString(e)); return DFTATOM_E_CUDA; }
    return 0;
}

// wide_from_step > 0: an atom whose SCF step counter has reached it is searched by the 8-warp shape (256 radial segments per orbital: half the
// depth of a round - the latency shape for the steps where few atoms are left), before that by the 4-warp shape (3 CTAs per SM: throughput); both are
// launched, the atom's own step counter decides (its records do not depend on what else is in the batch).  0: the 4-warp shape at every step.
int launch_search_rows(const GridDev& g, const double* atab, const AtomDev* atoms, const OrbitalDev* orbs, const AtomState* astate,
                       SearchState* ss, int n_orbs, unsigned long long* work, int warm_start, int cfg, int wide_from_step, int step_lo, int step_hi, cudaStream_t st)
{
    int n_launch = 0;
    // [step_lo, step_hi): the SCF steps this launch can be executed at (all atoms of a batch step together); a shape whose window misses it is not launched
    const int split = wide_from_step > 0 ? wide_from_step : (1 << 30);
    if (step_lo < split) {
        launch_step_kernel(search_rows_kernel<kRowWarps>, dim3(n_orbs), dim3(32 * kRowWarps), rows_smem_bytes(kRowWarps), st, g, atab, atoms, orbs, astate, ss, n_orbs, work, warm_start, cfg, 0, split);
        ++n_launch;
    }
    if (wide_from_step > 0 && step_hi > split) {
        launch_step_kernel(search_rows_kernel<kRowWarpsWide>, dim3(n_orbs), dim3(32 * kRowWarpsWide), rows_smem_bytes(kRowWarpsWide), st, g, atab, atoms, orbs, astate, ss, n_orbs,
                           work, warm_start, cfg, split, 1 << 30);
        ++n_launch;
    }
    return n_launch;
}

}  // namespace dft
