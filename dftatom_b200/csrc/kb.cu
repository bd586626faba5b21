// Kleinman-Bylander form of semilocal pseudopotentials and its logarithmic derivatives (dftatom_kb_form / dftatom_kb_log_derivatives,
// include/dftatom_b200.h).
//
// kb_form_kernel: one CTA per channel.  Threads stride over the nodes 0..i_s (a, b) and 0..N-1 (<u|u>); the partial sums are reduced
// in shared memory in a fixed tree order, so the result does not depend on scheduling.  Every thread then writes its nodes of beta.
//
// kb_proj_kernel: per projector the two rows the driven sweep reads, in the index variable of the sweep (y = u e^(-delta i / 2)):
// the Numerov source s_i = 2 K_i beta_i e^(-delta i / 2) of -1/2 u'' + (V - E) u = -beta (uniform grid: 2 h^2 beta_i), and the
// projection weight h_i = w_i beta_i (dr/di)_i e^(delta i / 2) (w_i the sweep rule on 0..i_s), so that <beta|u> = sum_i h_i y_i.
//
// kb_logderiv_kernel: one warp = 32 energies of one channel (warp-uniform table loads), warps dealt longest sweep first like
// logderiv_kernel.  A channel without projector runs logderiv_sweep itself.  A channel with one runs kb_sweep: the homogeneous chain
// u_h and the chain u_p driven by -beta in one lane, each rescaled on its own by exact powers of two (u_p together with the scale
// sigma of its source), then u = (sigma - E_KB h_p) u_h + E_KB h_h u_p in the final scale of both.  The node count needs the
// combination at every node 1..i_c, which is known only once h_h, h_p are: a second pass repeats both recurrences to i_c (same
// operations, so the same values and rescales) and counts the sign changes of the combination.
#include "logderiv_sweep.cuh"

namespace dft {

namespace {
constexpr int kKbThreads = 256;
__device__ __forceinline__ double kb_nan() { return __longlong_as_double(0x7ff8000000000000LL); }
}

__global__ void __launch_bounds__(kKbThreads) kb_form_kernel(GridDev g, KbFormArgs a)
{
    __shared__ double red[3][kKbThreads];
    const int c = blockIdx.x, N = g.N, t = threadIdx.x;
    const int row = a.row[c], loc = a.loc[c], is = a.is[c];
    const double* __restrict__ V = a.V + (size_t)row * N;
    const double* __restrict__ VL = a.V + (size_t)loc * N;
    const double* __restrict__ u = a.u + (size_t)row * N;
    const bool local = row == loc;
    double sa = 0., sb = 0., su = 0.;
    for (int i = t; i < N; i += kKbThreads) {
        const double ui = u[i];
        su = fma(g.wjac[i] * ui, ui, su);
        if (!local && i >= 1 && i <= is) {
            const double dv = V[i] - VL[i];
            const double jac = g.uniform ? g.h : g.rp * g.delta * g.ex[i];
            const double f = simpson_weight(i, is) * (ui * ui) * jac;
            sa = fma(f, dv, sa);
            sb = fma(f * dv, dv, sb);
        }
    }
    red[0][t] = sa; red[1][t] = sb; red[2][t] = su;
    __syncthreads();
    for (int s = kKbThreads / 2; s > 0; s >>= 1) {
        if (t < s) for (int q = 0; q < 3; ++q) red[q][t] += red[q][t + s];
        __syncthreads();
    }
    const double A = red[0][0], B = red[1][0], UU = red[2][0];
    const int status = local ? 1 : ((A == 0. || is < 3) ? 2 : 0);
    if (t == 0) {
        dftatom_kb_result* r = a.res + c;
        r->E_KB = status == 1 ? 0. : (status == 2 ? kb_nan() : B / A);
        r->cos = status == 1 ? 1. : (status == 2 ? kb_nan() : A / sqrt(UU * B));
        r->i_s = is; r->r_s = g.r[is]; r->status = status;
    }
    const double inv_sb = status == 0 ? 1. / sqrt(B) : 0.;
    double* __restrict__ beta = a.beta + (size_t)c * N;
    for (int i = t; i < N; i += kKbThreads)
        beta[i] = (status == 0 && i >= 1 && i <= is) ? (V[i] - VL[i]) * u[i] * inv_sb : 0.;
}

// source and projection rows of every projector (blockIdx.y)
__global__ void kb_proj_kernel(GridDev g, KbProjArgs a)
{
    const int p = blockIdx.y, N = g.N, is = a.is[p];
    const double* __restrict__ beta = a.beta + (size_t)p * N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        const double b = beta[i];
        double s, h;
        if (g.uniform) { s = g.k2[i] * b; h = g.h * b; }
        else { s = g.k2[i] * b / g.sqex[i]; h = (g.rp * g.delta) * g.ex[i] * g.sqex[i] * b; }
        a.src[(size_t)p * N + i] = s;
        a.hw[(size_t)p * N + i] = i <= is ? simpson_weight(i, is) * h : 0.;
    }
}

// The two chains of kb_sweep: homogeneous (h) and driven by -sigma beta (p), both y = u e^(-delta i / 2); one Numerov step to node i
struct KbChains {
    double yh, wh, whp, yp, wp, wpp;      // y, w and w of the node before, per chain
    double gq, sig, sm, s0;               // g at the current node; source scale; source at the node before and the current node
    double gprev;
    bool bad;
    __device__ __forceinline__ void step(double gi, double sp)
    {
        const double src3 = (fma(10., s0, sm) + sp) * (1. / 12.);
        const double wnh = fma(12. * gq, yh, fma(2., wh, -whp));
        const double wnp = fma(sig, src3, fma(12. * gq, yp, fma(2., wp, -wpp)));
        const double d = 1. - gi;
        bad |= !(d > 0.);
        const double rd = 1. / d;
        whp = wh; wh = wnh; wpp = wp; wp = wnp;
        gprev = gq; gq = gi; sm = s0; s0 = sp;
        yh = wnh * rd; yp = wnp * rd;
    }
};

// D, u, du and the node count at node n = i_c of the solution of -1/2 u'' + (V - E) u + E_KB beta <beta|u> = 0 regular at the nucleus;
// ns = i_s of the projector, `src` / `hw` its rows of kb_proj_kernel
__device__ __forceinline__ dftatom_logderiv kb_sweep(const GridDev& g, const double* __restrict__ atab, const double* __restrict__ src,
                                                  const double* __restrict__ hw, int l, int n, int ns, double E, double ekb)
{
    const double* __restrict__ b12 = g.b12;
    const double* __restrict__ c6 = g.c6;
    const double* __restrict__ k2 = g.k2;
    const double ll1 = (double)(l * (l + 1));
    auto gval = [&](int i) { return fma(-E, __ldg(c6 + i), fma(ll1, __ldg(b12 + i), __ldg(atab + i))); };
    const double y1 = g.uniform ? pow(g.h, (double)l + 1.) : pow(__ldg(g.r + 1), (double)l + 1.) * exp(-0.5 * g.delta);
    const int nmax = max(n, ns);
    auto init = [&](KbChains& q) {
        q.yh = y1; q.gq = gval(1); q.wh = (1. - q.gq) * y1; q.whp = 0.;
        q.yp = 0.; q.wp = 0.; q.wpp = 0.;
        q.sig = 1.; q.sm = __ldg(src); q.s0 = __ldg(src + 1); q.gprev = 0.; q.bad = false;
    };
    // pass 1: both chains to nmax + 1, the projections over 0..ns, the three norm sums over 0..n, y at n - 1, n, n + 1
    KbChains q;
    init(q);
    double hh = __ldg(hw + 1) * y1, hp = 0.;
    const double w1 = simpson_weight(1, n) * __ldg(k2 + 1);
    double Shh = w1 * y1 * y1, Shp = 0., Spp = 0.;
    double yh_m = y1, yp_m = 0., g_m = q.gq, yh_c = 0., yp_c = 0., yh_n = 0., yp_n = 0., g_n = 0., sg_m = __ldg(src + 1), sg_n = 0.;
    int eh = 0, ep = 0;
    for (int i = 2; i <= nmax + 1; ++i) {
        q.step(gval(i), __ldg(src + i));
        if (i <= ns) { const double hi = __ldg(hw + i); hh = fma(hi, q.yh, hh); hp = fma(hi, q.yp, hp); }
        if (i <= n) {
            const double wq = simpson_weight(i, n) * __ldg(k2 + i);
            Shh = fma(wq * q.yh, q.yh, Shh); Shp = fma(wq * q.yh, q.yp, Shp); Spp = fma(wq * q.yp, q.yp, Spp);
        }
        if (i == n - 1) { yh_m = q.yh; yp_m = q.yp; g_m = q.gq; sg_m = q.s0; }
        if (i == n) { yh_c = q.yh; yp_c = q.yp; }
        if (i == n + 1) { yh_n = q.yh; yp_n = q.yp; g_n = q.gq; sg_n = q.s0; }
        if ((i & 7) == 1) {                                  // every 8 nodes: exact rescale of either chain by a power of two
            if (fabs(q.yh) > kBig) {
                q.yh *= kDown; q.wh *= kDown; q.whp *= kDown; hh *= kDown; Shh *= kDown * kDown; Shp *= kDown;
                yh_m *= kDown; yh_c *= kDown; yh_n *= kDown; ++eh;
            }
            if (fabs(q.yp) > kBig) {
                q.yp *= kDown; q.wp *= kDown; q.wpp *= kDown; q.sig *= kDown; hp *= kDown; Spp *= kDown * kDown; Shp *= kDown;
                yp_m *= kDown; yp_c *= kDown; yp_n *= kDown; ++ep;
            }
        }
    }
    dftatom_logderiv o;
    o.pad = 0;
    if (q.bad) {
        o.D = o.u = o.du = kb_nan();
        o.nodes = -1;
        return o;
    }
    // u = A y_h + B y_p, both chains and sigma in their final scales
    const double sig = q.sig;
    const double A = fma(-ekb, hp, sig), B = ekb * hh;
    // pass 2: the same recurrences to node n; sign changes of the combination among its non-zero values at nodes 1..n.  At node i the
    // chains are 2^(256 dh) / 2^(256 dp) above their final scales (dh = eh - rescales so far): the combination's sign is that of
    // A y_h 2^(-256 (dh - dp)) + B y_p (dh >= dp), or A y_h + B y_p 2^(-256 (dp - dh))
    init(q);
    int dh = eh, dp = ep, count = 0, sgn = A > 0. ? 1 : (A < 0. ? -1 : 0), first = sgn;      // node 1 holds A y_1, y_1 > 0
    double f = ldexp(1., -256 * abs(dh - dp));
    for (int i = 2; i <= n; ++i) {
        q.step(gval(i), __ldg(src + i));
        if ((i & 7) == 1) {
            bool changed = false;
            if (fabs(q.yh) > kBig) { q.yh *= kDown; q.wh *= kDown; q.whp *= kDown; --dh; changed = true; }
            if (fabs(q.yp) > kBig) { q.yp *= kDown; q.wp *= kDown; q.wpp *= kDown; q.sig *= kDown; --dp; changed = true; }
            if (changed) f = ldexp(1., -256 * abs(dh - dp));
        }
        const double x = A * q.yh, z = B * q.yp;
        const double v = dh >= dp ? fma(x, f, z) : fma(z, f, x);
        const int s = v > 0. ? 1 : (v < 0. ? -1 : 0);
        if (s != 0) { if (sgn != 0 && s != sgn) ++count; sgn = s; if (first == 0) first = s; }
    }
    const double flip = first < 0 ? -1. : 1.;               // u > 0 next to the nucleus
    const double y_c = fma(A, yh_c, B * yp_c), y_m = fma(A, yh_m, B * yp_m), y_n = fma(A, yh_n, B * yp_n);
    // fourth-order index derivative with the source of the combination (B sigma s): y' = [(1 - 2 g_(n+1)) y_(n+1) - (1 - 2 g_(n-1)) y_(n-1)] / 2
    // - B sigma (s_(n+1) - s_(n-1)) / 12
    const double dy = fma(-B * sig, (sg_n - sg_m) * (1. / 12.), 0.5 * (fma(-2. * g_n, y_n, y_n) - fma(-2. * g_m, y_m, y_m)));
    const double s = fma(A * A, Shh, fma(2. * A * B, Shp, (B * B) * Spp));
    double uc, du, jac2;
    if (g.uniform) {
        uc = y_c; du = dy / g.h; jac2 = 2. * g.h;
    } else {
        const double sq = __ldg(g.sqex + n);
        uc = y_c * sq; du = fma(0.5 * g.delta, y_c, dy) / (sq * (g.rp * g.delta)); jac2 = 2. * (g.rp * g.delta);
    }
    const double inv_norm = flip / sqrt(s / jac2);
    o.D = du / uc; o.u = uc * inv_norm; o.du = du * inv_norm; o.nodes = count;
    return o;
}

__global__ void __launch_bounds__(128) kb_logderiv_kernel(GridDev g, KbLogDerivArgs a)
{
    const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (warp >= a.n_warps) return;
    const int item = a.warp_item[warp];
    const int ch = item / a.energy_blocks;
    const int e = (item - ch * a.energy_blocks) * 32 + (threadIdx.x & 31);
    const double E = a.E[min(e, a.n_energies - 1)];      // tail lanes repeat the last energy and write nothing
    const double* atab = a.atab + (size_t)a.pot[ch] * g.N;
    const int pj = a.proj[ch];
    const dftatom_logderiv o = pj < 0 ? logderiv_sweep(g, atab, a.l[ch], a.ic[ch], E)
                                      : kb_sweep(g, atab, a.src + (size_t)pj * g.N, a.hw + (size_t)pj * g.N, a.l[ch], a.ic[ch], a.is[pj], E,
                                                 a.ekb[ch]);
    if (e < a.n_energies) a.out[(size_t)ch * a.n_energies + e] = o;
}

void launch_kb_form(const GridDev& g, const KbFormArgs& a, cudaStream_t st)
{
    kb_form_kernel<<<a.n_channels, kKbThreads, 0, st>>>(g, a);
}

void launch_kb_proj(const GridDev& g, const KbProjArgs& a, cudaStream_t st)
{
    const int chunks = g.N > 64 * 1024 ? 64 : (g.N + 1023) / 1024;
    kb_proj_kernel<<<dim3(chunks, a.n_proj), 256, 0, st>>>(g, a);
}

void launch_kb_logderiv(const GridDev& g, const KbLogDerivArgs& a, cudaStream_t st)
{
    kb_logderiv_kernel<<<(a.n_warps + 3) / 4, 128, 0, st>>>(g, a);
}

}  // namespace dft
