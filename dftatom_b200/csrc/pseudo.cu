// Troullier-Martins pseudization of all-electron valence orbitals and unscreening to ionic potentials (dftatom_tm_pseudize,
// include/dftatom_b200.h).
//
// tm_kernel: one CTA of 8 warps per channel, CTAs dealt longest i_c first (the host orders `order`).  Warp 0 runs the outward sweep
// of dftatom_log_derivatives at E = eps (logderiv_sweep.cuh); thread 0 turns D, u_n(r_c) and V, V', V'' at r_c into the linear part
// of the coefficients.  In the scaled variable t = r / r_c with d_2k = c_2k r_c^2k and x = d_2 = c2 r_c^2, the p' .. p'''' conditions
// are M (d6, d8, d10, d12) = T - x e2 - d4 e4 with the constant integer matrix M_kj = P!/(P - k)! (P = 6, 8, 10, 12), so
// (d6 .. d12) = A + x B + x^2 C.  The norm F(x) = ln S(x) - ln q is evaluated by one warp per candidate x, the lanes striding over
// nodes 0..i_c; the ladder x = 0, -1/2, +1/2, -1, +1, ... is evaluated 8 candidates per round until the first interval (in the
// order of the definition) with a sign change, which 8-point multisection then shrinks to 1e-13 relative.
// tm_density_kernel / tm_unscreen_kernel: the valence density of each potential row and V_ion = V_scr - V_H - V_xc per channel.
// partial_core_kernel (dftatom_partial_core): the core density and its Louie-Froyen-Cohen partial core per row.
#include "logderiv_sweep.cuh"

namespace dft {

namespace {
constexpr int kTmWarps = 8;
constexpr int kLadder = 128;              // x = +-k/2, k = 0..kLadder
constexpr double kRelTol = 1e-13;
constexpr int kMaxRefine = 40;            // multisection rounds (each shrinks the bracket 9-fold: 1e-13 takes 15)
__device__ __forceinline__ double nan_value() { return __longlong_as_double(0x7ff8000000000000LL); }
}

// ladder candidate o (0, 1, 2, ...) -> x: 0, -1/2, +1/2, -1, +1, ...
__device__ __forceinline__ double ladder_x(int o) { return o == 0 ? 0. : ((o & 1) ? -0.5 * ((o + 1) >> 1) : 0.5 * (o >> 1)); }

// F at both ends of an interval changes sign (a zero counts; NaN never does)
__device__ __forceinline__ bool sign_change(double fa, double fb) { return (fa <= 0. && fb >= 0.) || (fa >= 0. && fb <= 0.); }

struct TmShared {
    double A[4], B[4], C[4];              // (d6 .. d12)(x) = A + x B + x^2 C
    double p0, inv_l5, lnq;               // ln(a / r_c^(l+1)), 1 / (2l + 5), ln q
    double xs[kTmWarps], F[kTmWarps];     // the candidates of one round and F there
    double Fl[2 * kLadder + 1];           // F on the ladder, index 2x + kLadder
    double lo, hi, flo, fhi;              // the bracket
    int state;                            // 0: scanning, 1: refining, 2: done, 3: failed (res->status says why)
};

// d0 .. d12 at x
__device__ __forceinline__ void tm_coeffs(const TmShared& s, double x, double d[7])
{
    d[1] = x;
    d[2] = -(x * x) * s.inv_l5;
    for (int k = 0; k < 4; ++k) d[3 + k] = fma(x, fma(x, s.C[k], s.B[k]), s.A[k]);
    d[0] = s.p0 - (((((d[1] + d[2]) + d[3]) + d[4]) + d[5]) + d[6]);
}

// p(t) = sum d_2k t^2k by Horner in t^2
__device__ __forceinline__ double tm_p(const double d[7], double t2)
{
    return fma(t2, fma(t2, fma(t2, fma(t2, fma(t2, fma(t2, d[6], d[5]), d[4]), d[3]), d[2]), d[1]), d[0]);
}

__device__ __forceinline__ double pow_l1(double r, int l) { double v = r; for (int k = 0; k < l; ++k) v *= r; return v; }

// ln S(x) - ln q, S = sum_i w_i r_i^(2l+2) e^(2 p(r_i)) (dr/di)_i over nodes 0..n, reduced over the warp
__device__ double tm_norm_F(const GridDev& g, const TmShared& s, double x, int l, int n, double inv_rc)
{
    double d[7];
    tm_coeffs(s, x, d);
    double acc = 0.;
    for (int i = (int)(threadIdx.x & 31); i <= n; i += 32) {
        const double r = __ldg(g.r + i);
        const double t = r * inv_rc;
        const double u = pow_l1(r, l) * exp(tm_p(d, t * t));
        const double jac = g.uniform ? g.h : g.rp * g.delta * __ldg(g.ex + i);
        acc = fma(simpson_weight(i, n) * u * u, jac, acc);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return log(acc) - s.lnq;
}

__global__ void __launch_bounds__(kTmWarps * 32) tm_kernel(GridDev g, TmArgs a)
{
    __shared__ TmShared s;
    const int c = a.order[blockIdx.x];
    const int N = g.N, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = a.pot[c], l = a.l[c], n = a.ic[c];
    const double eps = a.eps[c];
    const double* __restrict__ V = a.V + (size_t)p * N;
    const double* __restrict__ urow = a.u + (size_t)a.orbital[c] * N;
    const double rc = g.r[n], inv_rc = 1. / rc;
    dftatom_tm_result* res = a.res + c;
    if (warp == 0) {
        const dftatom_logderiv o = logderiv_sweep(g, a.atab + (size_t)p * N, l, n, eps);
        if (lane == 0) {
            const double ua = urow[n];
            const double aa = fabs(ua);
            const double q = o.nodes < 0 ? nan_value() : (aa * aa) / (o.u * o.u);
            res->r_c = rc; res->q = q; res->pad = 0;
            if (o.nodes < 0) {
                s.state = 3; res->status = 2;
            } else {
                s.state = 0;
                const double L1 = (double)(l + 1);
                // V' and V'' at r_c: 5-point differences in the index, chain rule with dr/di = J (d2r/di2 = delta J)
                const double vi1 = ((V[n - 2] - 8. * V[n - 1]) + (8. * V[n + 1] - V[n + 2])) / 12.;
                const double vi2 = (((-V[n - 2] + 16. * V[n - 1]) - 30. * V[n]) + (16. * V[n + 1] - V[n + 2])) / 12.;
                const double J = g.uniform ? g.h : g.delta * (rc + g.rp);
                const double v1 = vi1 / J, v2 = (vi2 - g.delta * vi1) / (J * J);
                const double r2 = rc * rc, r3 = r2 * rc;
                const double p1 = o.D - L1 / rc;
                const double p2 = 2. * (V[n] - eps) - 2. * L1 * p1 / rc - p1 * p1;
                const double p3 = 2. * v1 + 2. * L1 * p1 / r2 - 2. * L1 * p2 / rc - 2. * p1 * p2;
                const double p4 = 2. * v2 - 4. * L1 * p1 / r3 + 4. * L1 * p2 / r2 - 2. * L1 * p3 / rc - 2. * p2 * p2 - 2. * p1 * p3;
                // M X = [T, e2, e4]: T = r_c^k p^(k), e2 / e4 = the t-derivatives of t^2 / t^4 at t = 1
                double M[4][4] = { { 6., 8., 10., 12. }, { 30., 56., 90., 132. }, { 120., 336., 720., 1320. }, { 360., 1680., 5040., 11880. } };
                double R[4][3] = { { rc * p1, 2., 4. }, { r2 * p2, 2., 12. }, { r3 * p3, 0., 24. }, { r2 * r2 * p4, 0., 24. } };
                for (int k = 0; k < 4; ++k)
                    for (int j = k + 1; j < 4; ++j) {
                        const double f = M[j][k] / M[k][k];
                        for (int q2 = k; q2 < 4; ++q2) M[j][q2] -= f * M[k][q2];
                        for (int q2 = 0; q2 < 3; ++q2) R[j][q2] -= f * R[k][q2];
                    }
                for (int k = 3; k >= 0; --k)
                    for (int q2 = 0; q2 < 3; ++q2) {
                        double v = R[k][q2];
                        for (int j = k + 1; j < 4; ++j) v -= M[k][j] * R[j][q2];
                        R[k][q2] = v / M[k][k];
                    }
                s.inv_l5 = 1. / (2. * l + 5.);
                for (int k = 0; k < 4; ++k) { s.A[k] = R[k][0]; s.B[k] = -R[k][1]; s.C[k] = R[k][2] * s.inv_l5; }
                s.p0 = log(aa / pow_l1(rc, l));
                s.lnq = log(q);
            }
        }
    }
    __syncthreads();
    // the ladder, kTmWarps candidates per round, in the order 0, -1/2, +1/2, -1, ...; intervals checked as the definition orders them
    int next = 1;                          // next interval: k = (next + 1) / 2, negative for odd next
    for (int base = 0; s.state == 0; base += kTmWarps) {
        const int o = base + warp;
        if (o <= 2 * kLadder) {
            const double x = ladder_x(o);
            const double F = tm_norm_F(g, s, x, l, n, inv_rc);
            if (lane == 0) s.Fl[(int)(2. * x) + kLadder] = F;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int evaluated = min(base + kTmWarps, 2 * kLadder + 1);
            for (; next <= 2 * kLadder && next < evaluated && s.state == 0; ++next) {
                const int k = (next + 1) >> 1;
                const bool neg = next & 1;
                const double xa = neg ? -0.5 * k : 0.5 * (k - 1), xb = neg ? -0.5 * (k - 1) : 0.5 * k;
                const double fa = s.Fl[(int)(2. * xa) + kLadder], fb = s.Fl[(int)(2. * xb) + kLadder];
                if (sign_change(fa, fb)) { s.lo = xa; s.hi = xb; s.flo = fa; s.fhi = fb; s.state = 1; }
            }
            if (s.state == 0 && next > 2 * kLadder) { s.state = 3; res->status = 1; }
        }
        __syncthreads();
    }
    // multisection: kTmWarps interior points per round; the sub-interval nearest x = 0 with a sign change is kept
    for (int round = 0; s.state == 1; ++round) {
        const double lo = s.lo, hi = s.hi;
        const double x = lo + (hi - lo) * ((double)(warp + 1) * (1. / (kTmWarps + 1)));
        const double F = tm_norm_F(g, s, x, l, n, inv_rc);
        if (lane == 0) { s.xs[warp] = x; s.F[warp] = F; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double xv[kTmWarps + 2], fv[kTmWarps + 2];
            xv[0] = lo; fv[0] = s.flo; xv[kTmWarps + 1] = hi; fv[kTmWarps + 1] = s.fhi;
            for (int j = 0; j < kTmWarps; ++j) { xv[j + 1] = s.xs[j]; fv[j + 1] = s.F[j]; }
            const bool neg = hi <= 0.;
            for (int j = 0; j <= kTmWarps; ++j) {
                const int k = neg ? kTmWarps - j : j;
                if (sign_change(fv[k], fv[k + 1])) { s.lo = xv[k]; s.hi = xv[k + 1]; s.flo = fv[k]; s.fhi = fv[k + 1]; break; }
            }
            if (s.hi - s.lo <= kRelTol * fmax(fabs(s.lo), fabs(s.hi))) {
                s.state = 2; res->status = 0;
            } else if (round + 1 >= kMaxRefine || (s.lo == lo && s.hi == hi)) {      // no sub-interval changed sign, or out of rounds
                s.state = 3; res->status = 3;
            }
        }
        __syncthreads();
    }
    // the rows: r^(l+1) e^p and eps + [p'' + p'^2 + 2(l+1) p'/r] / 2 inside r_c, the all-electron rows beyond
    double d[7];
    const bool ok = s.state == 2;
    if (ok) tm_coeffs(s, 0.5 * (s.lo + s.hi), d);
    else for (int k = 0; k < 7; ++k) d[k] = nan_value();
    if (threadIdx.x == 0) {
        double sc = 1.;
        for (int k = 0; k < 7; ++k) { res->c[k] = d[k] / sc; sc *= rc * rc; }
    }
    const double sgn = urow[n] < 0. ? -1. : 1.;
    const double inv_rc2 = inv_rc * inv_rc, L1 = (double)(l + 1);
    double* __restrict__ up = a.u_ps + (size_t)c * N;
    double* __restrict__ vs = a.v_scr + (size_t)c * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        double uo, vo;
        if (i == 0) {
            uo = 0.; vo = 0.;
        } else if (i <= n) {
            const double r = g.r[i];
            const double t = r * inv_rc, t2 = t * t;
            uo = pow_l1(r, l) * exp(tm_p(d, t2));
            // p'/r and p'' as polynomials in t^2 (times 1 / r_c^2)
            const double q = inv_rc2 * fma(t2, fma(t2, fma(t2, fma(t2, fma(t2, 12. * d[6], 10. * d[5]), 8. * d[4]), 6. * d[3]), 4. * d[2]), 2. * d[1]);
            const double p2 = inv_rc2 * fma(t2, fma(t2, fma(t2, fma(t2, fma(t2, 132. * d[6], 90. * d[5]), 56. * d[4]), 30. * d[3]), 12. * d[2]), 2. * d[1]);
            vo = eps + 0.5 * ((p2 + (r * r) * (q * q)) + 2. * L1 * q);
        } else {
            uo = sgn * urow[i]; vo = V[i];
        }
        up[i] = uo; vs[i] = vo;
    }
}

// valence density of each potential row: rho_v = sum occ u_ps^2 / (4 pi r^2), 0 where a channel of the row failed
__global__ void tm_density_kernel(GridDev g, TmRowArgs a)
{
    const int p = blockIdx.y, N = g.N;
    const int c0 = a.row_begin[p], c1 = a.row_begin[p + 1];
    bool failed = false;
    for (int k = c0; k < c1; ++k) failed |= a.res[a.row_chan[k]].status != 0;
    double* __restrict__ rho = a.rho + (size_t)a.slot[p] * N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        double acc = 0.;
        if (!failed)
            for (int k = c0; k < c1; ++k) {
                const int c = a.row_chan[k];
                const double u = a.u_ps[(size_t)c * N + i];
                acc = fma(a.occ[c] * u, u, acc);
            }
        rho[i] = acc * g.inv4pr2[i];
    }
}

// V_ion = V_scr - U / r - V_xc per channel (blockIdx.y < n_channels) and the valence density per row (the rest); NaN (nodes 1..N-1)
// for a row with a failed channel
__global__ void tm_unscreen_kernel(GridDev g, TmRowArgs a)
{
    const int y = blockIdx.y, N = g.N;
    const bool chan = y < a.n_channels;
    const int p = chan ? a.pot[y] : y - a.n_channels;
    bool failed = false;
    for (int k = a.row_begin[p]; k < a.row_begin[p + 1]; ++k) failed |= a.res[a.row_chan[k]].status != 0;
    const int sl = a.slot[p];
    const double* __restrict__ rho = a.rho + (size_t)sl * N;
    const double* __restrict__ vxc = a.vxc + (size_t)sl * N;
    const double* __restrict__ U = sl < a.n_solve ? a.U + (size_t)sl * a.ldU : nullptr;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
        if (chan) {
            double v = 0.;
            if (i > 0) v = failed ? nan_value() : (a.v_scr[(size_t)y * N + i] - (U ? U[i] / g.r[i] : 0.)) - vxc[i];
            a.v_ion[(size_t)y * N + i] = v;
        } else {
            a.rho_out[(size_t)p * N + i] = (failed && i > 0) ? nan_value() : rho[i];
        }
    }
}

// Louie-Froyen-Cohen partial core (dftatom_partial_core): one CTA per row.  The threads build rho_core = sum occ u^2 / (4 pi r^2) over
// the row's core entries at nodes 1..N-2; thread 0 takes the 5-point index derivative at i_pc, t = 1 + r rho' / rho, and the root x of
// x cos x - t sin x on (0, pi) by bisection to the last bit; then every thread writes its nodes of rho_pc, and n_core / n_pc are reduced
// in shared memory in a fixed tree order.
constexpr int kPcThreads = 256;
__global__ void __launch_bounds__(kPcThreads) partial_core_kernel(GridDev g, PcArgs a)
{
    __shared__ double red[2][kPcThreads];
    __shared__ double sA, sB;
    __shared__ int s_ok;
    const int p = blockIdx.x, N = g.N, t = threadIdx.x;
    const int e0 = a.core_begin[p], e1 = a.core_begin[p + 1], ipc = a.ipc[p];
    double* __restrict__ rc = a.rho_core + (size_t)p * N;
    double* __restrict__ rpc = a.rho_pc + (size_t)p * N;
    for (int i = t; i < N; i += kPcThreads) {
        double acc = 0.;
        if (i >= 1 && i <= N - 2)
            for (int k = e0; k < e1; ++k) {
                const double u = a.u[(size_t)a.core_orb[k] * N + i];
                acc = fma(a.core_occ[k] * u, u, acc);
            }
        rc[i] = acc * g.inv4pr2[i];
    }
    __syncthreads();                      // rho_core is read back below by other threads of the CTA
    if (t == 0) {
        dftatom_pcc_result* res = a.res + p;
        double A = 0., B = 0.;
        int ok = 1;
        if (ipc > 0) {
            const double r = g.r[ipc], rho = rc[ipc];
            const double di = ((rc[ipc - 2] - 8. * rc[ipc - 1]) + (8. * rc[ipc + 1] - rc[ipc + 2])) / 12.;
            const double J = g.uniform ? g.h : g.delta * (r + g.rp);
            const double tt = 1. + r * (di / J) / rho;
            ok = rho > 0. && tt < 1.;
            if (ok) {
                // x cot x falls from 1 to -inf on (0, pi): f = x cos x - t sin x is > 0 left of the root, < 0 right of it
                double lo = 0., hi = 3.14159265358979323846;
                for (int it = 0; it < 2000; ++it) {
                    const double mid = 0.5 * (lo + hi);
                    if (mid <= lo || mid >= hi) break;
                    if (mid * cos(mid) - tt * sin(mid) > 0.) lo = mid; else hi = mid;
                }
                const double x = 0.5 * (lo + hi);
                B = x / r; A = rho * r / sin(x);
            } else {
                A = nan_value(); B = nan_value();
            }
            res->r_pc = r;
        } else {
            res->r_pc = 0.;
        }
        res->A = A; res->B = B; res->i_pc = ipc; res->status = ok ? 0 : 1;
        sA = A; sB = B; s_ok = ok;
    }
    __syncthreads();
    const double A = sA, B = sB;
    const bool ok = s_ok;
    double nc = 0., np = 0.;
    for (int i = t; i < N; i += kPcThreads) {
        const double c = rc[i];
        double v;
        if (i == 0) v = 0.;
        else if (!ok) v = nan_value();
        else if (i < ipc) { const double r = g.r[i]; v = A * sin(B * r) / r; }
        else v = c;
        rpc[i] = v;
        const double w = g.wjac[i] * (4. * 3.14159265358979323846) * (g.r[i] * g.r[i]);
        nc = fma(w, c, nc);
        np = fma(w, v, np);
    }
    red[0][t] = nc; red[1][t] = np;
    __syncthreads();
    for (int s = kPcThreads / 2; s > 0; s >>= 1) {
        if (t < s) { red[0][t] += red[0][t + s]; red[1][t] += red[1][t + s]; }
        __syncthreads();
    }
    if (t == 0) { a.res[p].n_core = red[0][0]; a.res[p].n_pc = red[1][0]; a.res[p].pad = 0; }
}

// the xc argument of the core-corrected unscreening: out[slot[p]] = rho[slot[p]] + rho_pc[p] per potential row (blockIdx.y)
__global__ void core_xc_density_kernel(int N, const int* slot, const double* rho, const double* rho_pc, double* out)
{
    const int p = blockIdx.y;
    const size_t s = (size_t)slot[p] * N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) out[s + i] = rho[s + i] + rho_pc[(size_t)p * N + i];
}

void launch_partial_core(const GridDev& g, const PcArgs& a, cudaStream_t st)
{
    partial_core_kernel<<<a.n_rows, kPcThreads, 0, st>>>(g, a);
}

void launch_tm(const GridDev& g, const TmArgs& a, cudaStream_t st)
{
    tm_kernel<<<a.n_channels, kTmWarps * 32, 0, st>>>(g, a);
}

static int tm_row_chunks(int N) { const int c = (N + 1023) / 1024; return c > 64 ? 64 : c; }

void launch_tm_density(const GridDev& g, const TmRowArgs& a, cudaStream_t st)
{
    tm_density_kernel<<<dim3(tm_row_chunks(g.N), a.n_pot), 256, 0, st>>>(g, a);
}

void launch_tm_unscreen(const GridDev& g, const TmRowArgs& a, cudaStream_t st)
{
    tm_unscreen_kernel<<<dim3(tm_row_chunks(g.N), a.n_channels + a.n_pot), 256, 0, st>>>(g, a);
}

void launch_core_xc_density(const GridDev& g, int n_pot, const int* slot, const double* rho, const double* rho_pc, double* rho_xc, cudaStream_t st)
{
    core_xc_density_kernel<<<dim3(tm_row_chunks(g.N), n_pot), 256, 0, st>>>(g.N, slot, rho, rho_pc, rho_xc);
}

}  // namespace dft
