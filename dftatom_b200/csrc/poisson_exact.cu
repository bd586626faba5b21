// Bit-reproducible radial Poisson multigrid ("poisson_exact" mode): the reference's FullCycle in the reference's own
// floating-point expression order, without FMA contraction, with its data-dependent early exits and its 100 V-cycles, so
// that U(r) equals the CPU reference's PhiLevels[0] BIT FOR BIT.
//
// Replaces (reference DFTAtom/) PoissonSolver.h:51-81 SolvePoissonNonUniform / :20-49 SolvePoissonUniform, :89-124 FullCycle,
// :155-159 VCycle, PoissonSolver.cpp:40-64 GaussSeidel, :66-77 IterateGaussSeidel, :80-106 Initialize, :110-123 Prolong,
// :126-157 Restrict, :162-197 Ascend/Descend.
//
// Why it exists.  The plain FP64 multigrid of the reference stalls on a rounding floor whose offset from the exact discrete
// solution is a property of the exact operation order (worth 1e-5 .. 3e-4 Ha in the energies on the 65537- and 131073-node
// grids).  The production solver (poisson.cu: FMA, truncated affine scans, 8 V-cycles, warm start) lands on a different
// point of that floor; this kernel lands on the reference's.  It is a validation / parity mode: one CTA per density, every
// level in global memory (L2), no attempt at speed beyond running the chunks of a sweep concurrently.
//
// How a lexicographic Gauss-Seidel sweep is run in parallel and still bit-identical: the sweep is the first-order recurrence
//     Phi_i <- 0.5 (S_i + Phi_{i-1}^new + Phi_{i+1}^old - d_l (Phi_{i+1}^old - Phi_{i-1}^new) 0.5),
// whose dependence on the left neighbour contracts by a = (1 + d_l/2)/2 <= 0.508 per node on every level with >= 256
// intervals.  A thread that owns the nodes [s, s + C) starts kHalo = 128 nodes to the left from the OLD value of node
// s - 129 instead of the new one: the error of that start value decays by a^128 < 3e-38 before the first owned node,
// i.e. far below half an ulp of anything it is added to, and from there on the thread executes exactly the operations the
// serial sweep executes on exactly the same operands.  Sweeps are out of place (old -> new buffer), so no thread reads a
// value another thread is overwriting.  Levels with < 256 intervals are swept serially by one thread.
#include "internal.h"
#include <cmath>

namespace dft {

constexpr int kXT = 1024;      // threads per CTA
constexpr int kXHalo = 128;    // warm-up nodes; also the minimum chunk of a parallel level
constexpr int kXSerialBelow = 256;   // levels with fewer intervals run on one thread

struct XLevel {
    int n;          // intervals: nodes 0..n, node 0 / n are the boundaries
    int lgC, T;     // owner-major layout: T threads x C = 2^lgC consecutive nodes; node i -> slot (i mod C) T + i / C, node n -> slot n
    int off;        // offset of the level inside one buffer
    double d;       // deltaGridLevel[l]   (PoissonSolver.cpp:21-26)
};

struct XShared {
    XLevel lv[24];
    double red[32];
    double bcast;
    unsigned parity;     // bit l: the current Phi of level l lives in buffer B
};
__shared__ XShared xs;

__device__ __forceinline__ int xslot(const XLevel& v, int i)
{
    return i >= v.n ? v.n : ((i & ((1 << v.lgC) - 1)) * v.T + (i >> v.lgC));
}

__host__ __device__ inline void xlevel_geometry(int n, int* lgC, int* T)
{
    int t = 1;
    if (n >= kXSerialBelow) { t = n / kXHalo; if (t > kXT) t = kXT; }
    int c = n / t, lg = 0;
    while ((1 << lg) < c) ++lg;
    *lgC = lg; *T = t;
}

__host__ __device__ inline long long exact_level_total(int L)
{
    long long off = 0;
    for (int l = 0; l < L; ++l) off += (((1ll << (L - l)) + 1) + 3) & ~3ll;
    return off;
}
long long exact_poisson_work_doubles(int L) { return 3 * exact_level_total(L); }

__device__ __forceinline__ double x_block_sum(double v)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) xs.red[w] = v;
    __syncthreads();
    if (w == 0) {
        double t = xs.red[lane];
#pragma unroll
        for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) xs.bcast = t;
    }
    __syncthreads();
    return xs.bcast;
}

// one Gauss-Seidel update in the reference's operation order (PoissonSolver.cpp:56-57); no contraction
__device__ __forceinline__ double x_update(double s, double pm, double pp, double d)
{
    const double t1 = __dadd_rn(__dadd_rn(s, pm), pp);
    const double t2 = __dmul_rn(__dmul_rn(d, __dsub_rn(pp, pm)), 0.5);
    return __dmul_rn(0.5, __dsub_rn(t1, t2));
}

struct XBuf { double* A; double* B; double* S; };
__device__ __forceinline__ double* x_cur(const XBuf& b, int l) { return (((xs.parity >> l) & 1u) ? b.B : b.A) + xs.lv[l].off; }
__device__ __forceinline__ double* x_nxt(const XBuf& b, int l) { return (((xs.parity >> l) & 1u) ? b.A : b.B) + xs.lv[l].off; }

// GaussSeidel(lvl): returns sqrt(sum (old - new)^2), block-uniform
__device__ double x_sweep(const XBuf& b, int l)
{
    const XLevel v = xs.lv[l];
    const double* cur = x_cur(b, l);
    double* nxt = x_nxt(b, l);
    const double* src = b.S + v.off;
    const int t = threadIdx.x, C = 1 << v.lgC, T = v.T;
    double acc = 0.;
    if (t < T) {
        const double d = v.d;
        const int s = t * C;
        double pm;
        if (t == 0) {
            pm = cur[0];
            nxt[0] = pm;                                    // boundaries are never updated
        } else {
            int i = s - kXHalo;                             // warm-up over the last kXHalo nodes of the left neighbour (C >= kXHalo)
            if (i < 1) i = 1;
            pm = cur[xslot(v, i - 1)];                      // old value (or the boundary itself): its error has decayed by the time node s is reached
            for (; i < s; ++i) pm = x_update(src[xslot(v, i)], pm, cur[xslot(v, i + 1)], d);
        }
        // owned nodes: k-th node at slot k T + t
        const int k0 = (t == 0) ? 1 : 0;
        double pc = cur[k0 * T + t];
        for (int k = k0; k < C; ++k) {
            const int i = s + k;
            if (i >= v.n) break;
            const double pp = (k + 1 < C) ? cur[(k + 1) * T + t] : cur[xslot(v, i + 1)];
            const double x = x_update(src[k * T + t], pm, pp, d);
            nxt[k * T + t] = x;
            const double dif = __dsub_rn(pc, x);
            acc = __dadd_rn(acc, __dmul_rn(dif, dif));
            pm = x;
            pc = pp;
        }
        if (t == T - 1) nxt[v.n] = cur[v.n];
    }
    const double tot = x_block_sum(acc);
    if (threadIdx.x == 0) xs.parity ^= (1u << l);
    __syncthreads();
    return sqrt(tot);
}

// IterateGaussSeidel (.cpp:66-77)
__device__ double x_smooth(const XBuf& b, int l, double tol, int sweeps)
{
    double err = 1e10;
    for (int k = 0; k < sweeps; ++k) { err = x_sweep(b, l); if (err < tol) break; }
    return err;
}

// Restrict(l) (.cpp:126-157): Phi_l = 0, Source_l = 4 (injected residual of level l-1) - d_l (first difference)
__device__ void x_restrict_to(const XBuf& b, int l)
{
    const XLevel vf = xs.lv[l - 1], vc = xs.lv[l];
    const double* pf = x_cur(b, l - 1);
    const double* sf = b.S + vf.off;
    double* pc = x_cur(b, l);
    double* sc = b.S + vc.off;
    for (int i = threadIdx.x; i <= vc.n; i += kXT) {
        const int sl = xslot(vc, i);
        pc[sl] = 0.;
        if (i == 0 || i == vc.n) { sc[sl] = 0.; continue; }
        const int k = 2 * i;
        const double pm = pf[xslot(vf, k - 1)], p0 = pf[xslot(vf, k)], pp = pf[xslot(vf, k + 1)];
        const double lap = __dadd_rn(__dsub_rn(__dadd_rn(sf[xslot(vf, k)], pm), __dmul_rn(2., p0)), pp);
        sc[sl] = __dsub_rn(__dmul_rn(4., lap), __dmul_rn(vc.d, __dsub_rn(pp, pm)));
    }
    __syncthreads();
}

// Prolong(Phi_l -> Phi_{l-1}) (.cpp:110-123)
__device__ void x_prolong_from(const XBuf& b, int l)
{
    const XLevel vf = xs.lv[l - 1], vc = xs.lv[l];
    const double* pc = x_cur(b, l);
    double* pf = x_cur(b, l - 1);
    for (int i = threadIdx.x; i <= vc.n; i += kXT) {
        const double c = pc[xslot(vc, i)];
        const int s2 = xslot(vf, 2 * i);
        pf[s2] = __dadd_rn(pf[s2], c);
        if (i >= 1) {
            const int s1 = xslot(vf, 2 * i - 1);
            pf[s1] = __dadd_rn(pf[s1], __dmul_rn(0.5, __dadd_rn(pc[xslot(vc, i - 1)], c)));
        }
    }
    __syncthreads();
}

__device__ void x_to_coarse(const XBuf& b, int from, int to, double tol, int sweeps)
{   // Ascend (.cpp:162-171)
    for (int l = from; l < to;) { x_smooth(b, l, tol, sweeps); x_restrict_to(b, ++l); }
    x_smooth(b, to, tol, sweeps);
}
__device__ double x_to_fine(const XBuf& b, int from, int to, double tol, int sweeps)
{   // Descend (.cpp:173-186)
    double err = 1e10;
    for (int l = from; l > to; --l) { x_prolong_from(b, l); err = x_smooth(b, l - 1, tol, sweeps); }
    return err;
}

__global__ void __launch_bounds__(kXT, 1) poisson_exact_kernel(ExactPoissonArgs a)
{
    const int k = blockIdx.x;
    if (a.skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(a.skip) + (size_t)k * a.skip_stride_bytes)) return;
    const int L = a.L, c = L - 1;
    if (threadIdx.x == 0) {
        int off = 0;
        double d = a.delta;
        for (int l = 0; l < L; ++l) {
            XLevel v; v.n = 1 << (L - l); xlevel_geometry(v.n, &v.lgC, &v.T); v.off = off; v.d = d;
            xs.lv[l] = v;
            off += (v.n + 1 + 3) & ~3;
            d = __dmul_rn(d, 2.);
        }
        xs.parity = 0u;
    }
    __syncthreads();
    const long long tot = exact_level_total(L);
    XBuf b;
    b.A = a.work + (size_t)k * 3 * tot; b.B = b.A + tot; b.S = b.B + tot;
    const double* rho = a.rho + (size_t)k * a.rho_stride;
    const double hi_bc = a.Zbc[k];

    // Source_0 (PoissonSolver.h:55-74 / :22-43) and Initialize (.cpp:80-106)
    {
        const XLevel v0 = xs.lv[0];
        for (int i = threadIdx.x; i <= v0.n; i += kXT) {
            const int sl = xslot(v0, i);
            b.A[v0.off + sl] = 0.;
            b.S[v0.off + sl] = (i >= 1 && i < v0.n) ? __dmul_rn(a.r[i], __dmul_rn(a.pex[i], rho[i])) : 0.;
        }
        __syncthreads();
        for (int l = 1; l < L; ++l) {
            const XLevel vf = xs.lv[l - 1], vc = xs.lv[l];
            for (int p = threadIdx.x; p <= vc.n; p += kXT) {
                const int sl = xslot(vc, p);
                b.A[vc.off + sl] = 0.;
                b.S[vc.off + sl] = (p >= 1 && p < vc.n) ? __dmul_rn(4., b.S[vf.off + xslot(vf, 2 * p)]) : 0.;
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) { const XLevel vc = xs.lv[c]; b.A[vc.off + 0] = 0.; b.A[vc.off + vc.n] = hi_bc; }
        __syncthreads();
    }
    const double tol = 1e-3, tol_last = 1e-14;
    const int sweeps = 3;
    x_smooth(b, c, tol, 15);
    // FullCycle (PoissonSolver.h:89-124)
    for (int l = L - 2; l > 0; --l) {
        x_to_fine(b, c, l, tol, sweeps);
        x_to_coarse(b, l, c, tol, sweeps);
    }
    x_to_fine(b, c, 0, tol_last, sweeps);
    int used = 0;
    for (; used < a.max_vcycles; ++used) {
        x_to_coarse(b, 0, c, tol_last, sweeps);
        const double err = x_to_fine(b, c, 0, tol_last, sweeps);
        if (err < tol_last) { ++used; break; }
    }
    if (a.vcycles_used && threadIdx.x == 0) a.vcycles_used[k] = used;
    // U(r) = PhiLevels[0], natural node order
    {
        const XLevel v0 = xs.lv[0];
        const double* p0 = x_cur(b, 0);
        double* U = a.U + (size_t)k * a.ldU;
        for (int i = threadIdx.x; i <= v0.n; i += kXT) U[i] = p0[xslot(v0, i)];
    }
}

void launch_poisson_exact(const ExactPoissonArgs& a, cudaStream_t st)
{
    poisson_exact_kernel<<<a.n_dens, kXT, 0, st>>>(a);
}

}  // namespace dft
