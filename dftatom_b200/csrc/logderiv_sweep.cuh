// The outward sweep of dftatom_log_derivatives (include/dftatom_b200.h) for one energy: shared by logderiv_kernel (one lane per energy)
// and tm_kernel (pseudo.cu: the all-electron data at r_c at the channel's eigenvalue).
//
// Started and stepped like numerov_lanes_outward_kernel (numerov.cu): g_i = f_i / 12 = atab_i + l(l+1) b12_i - E c6_i, y_0 = 0,
// y_1 = r_1^(l+1) e^(-delta/2) (uniform grid: h^(l+1)), w = (1 - g) y, w_(i+1) = 2 w_i - w_(i-1) + 12 g_i y_i, y = w / (1 - g).
// The sweep does not stop at turning points: it runs to i_c + 1 (the nearest node to r_c and one beyond, for the derivative).
// The norm integral is folded into the sweep (Simpson 1/3 as odd and even sums, the 3/8 rule on the last three intervals when i_c is
// odd), and the running state is rescaled by 2^-256 (exact) whenever |y| passes 2^128 at the end of an 8-node block; the norm sum is
// scaled by 2^-512 with it.
#pragma once
#include "internal.h"

namespace dft {

namespace {
constexpr double kBig = 0x1p128;       // rescale threshold of |y|, checked every 8 nodes
constexpr double kDown = 0x1p-256;     // scale of y and w at a rescale (the norm sum takes its square)
}

// Simpson weight of node i of 0..n (1/3 rule on 0..m, the 3/8 rule on m..n when n is odd), the rule of the sweep's norm
__device__ __forceinline__ double simpson_weight(int i, int n)
{
    const int m = (n & 1) ? n - 3 : n;
    double w = 0.;
    if (m > 0 && i <= m) w = (i == 0 || i == m) ? 1. / 3. : ((i & 1) ? 4. / 3. : 2. / 3.);
    if ((n & 1) && i >= m) w += (i == m || i == n) ? 0.375 : 1.125;
    return w;
}

// D, u, du and the node count at node n = i_c of the outward solution at energy E on the a-table row `atab`; nodes = -1 and NaN in
// D, u, du when 1 - g <= 0 at some node 2..n+1
__device__ __forceinline__ dftatom_logderiv logderiv_sweep(const GridDev& g, const double* __restrict__ atab, int l, int n, double E)
{
    const double* __restrict__ b12 = g.b12;
    const double* __restrict__ c6 = g.c6;
    const double* __restrict__ k2 = g.k2;
    const int m = (n & 1) ? n - 3 : n;                    // Simpson 1/3 on 0..m, the 3/8 rule on m..n when n is odd
    const double ll1 = (double)(l * (l + 1));
    auto gval = [&](int i) { return fma(-E, __ldg(c6 + i), fma(ll1, __ldg(b12 + i), __ldg(atab + i))); };

    double y = g.uniform ? pow(g.h, (double)l + 1.) : pow(__ldg(g.r + 1), (double)l + 1.) * exp(-0.5 * g.delta);
    double gq = gval(1);
    double wprev = 0., w = (1. - gq) * y;
    double yprev = 0., gprev = 0.;
    bool positive = true, bad = false;                    // y_1 > 0; node 1 is exempt from the 1 - g > 0 test
    int count = 0;
    // one Numerov step to node i; `count_it`: node i is one of 1..i_c whose sign changes are counted
    auto step = [&](int i, bool count_it) {
        const double gi = gval(i);
        const double wn = fma(12. * gq, y, fma(2., w, -wprev));
        wprev = w; w = wn;
        const double d = 1. - gi;
        bad |= !(d > 0.);
        yprev = y; gprev = gq;
        y = wn / d; gq = gi;
        if (count_it && ((positive && y < 0.) || (!positive && y > 0.))) { ++count; positive = !positive; }
    };
    // f_i = y_i^2 k2_i = u_i^2 (dr/di) x 2 Rp delta (uniform grid: x 2 h); the constant is applied at the end
    const double f1 = y * y * __ldg(k2 + 1);
    double s_odd = m >= 2 ? f1 : 0., s_even = 0.;
    int i = 2;
    for (; i + 1 < m; i += 2) {                           // pairs (even i, odd i + 1) up to node m - 1
        step(i, true);
        s_even = fma(y * y, __ldg(k2 + i), s_even);
        step(i + 1, true);
        s_odd = fma(y * y, __ldg(k2 + i + 1), s_odd);
        if ((i & 6) == 0 && fabs(y) > kBig) {             // every 4th pair: exact rescale by a power of two
            y *= kDown; w *= kDown; wprev *= kDown;
            s_odd *= kDown * kDown; s_even *= kDown * kDown;
        }
    }
    // nodes m..n (f at m, and for odd n at m+1..m+3), then node n + 1
    double fm0 = 0., fm1 = 0., fm2 = 0., fm3 = 0.;       // f at nodes m .. m + 3
    auto fstep = [&](int j) { step(j, true); return y * y * __ldg(k2 + j); };
    if (m == 0) {                                         // n = 3: the 3/8 rule on 0..3 alone
        fm1 = f1; fm2 = fstep(2); fm3 = fstep(3);
    } else {
        fm0 = fstep(m);
        if (n & 1) { fm1 = fstep(m + 1); fm2 = fstep(m + 2); fm3 = fstep(m + 3); }
    }
    const double y_n = y, y_m1 = yprev, g_m1 = gprev;
    step(n + 1, false);
    dftatom_logderiv o;
    o.pad = 0;
    if (bad) {
        o.D = o.u = o.du = __longlong_as_double(0x7ff8000000000000LL);
        o.nodes = -1;
    } else {
        double s = (fm0 + 4. * s_odd + 2. * s_even) * (1. / 3.);
        if (n & 1) s += 0.375 * (fm0 + 3. * fm1 + 3. * fm2 + fm3);
        // fourth-order derivative on the index grid: y' = [(1 - 2 g_(n+1)) y_(n+1) - (1 - 2 g_(n-1)) y_(n-1)] / 2
        const double dy = 0.5 * (fma(-2. * gq, y, y) - fma(-2. * g_m1, y_m1, y_m1));
        double uc, du, jac2;                              // jac2 = 2 dr/di at node 0's scale: int u^2 dr = s / jac2
        if (g.uniform) {
            uc = y_n; du = dy / g.h; jac2 = 2. * g.h;
        } else {                                          // u = y e^(delta i / 2): u' = e^(-delta i / 2) (y' + delta y / 2) / (Rp delta)
            const double sq = __ldg(g.sqex + n);
            uc = y_n * sq; du = fma(0.5 * g.delta, y_n, dy) / (sq * (g.rp * g.delta)); jac2 = 2. * (g.rp * g.delta);
        }
        const double inv_norm = 1. / sqrt(s / jac2);
        o.D = du / uc; o.u = uc * inv_norm; o.du = du * inv_norm; o.nodes = count;
    }
    return o;
}

}  // namespace dft
