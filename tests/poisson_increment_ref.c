/* TEST INFRASTRUCTURE: the exact solution of the linear system of one warm Poisson solve in increment form (dftatom_poisson_increment),
 *     -a dU_{i-1} + dU_i - b dU_{i+1} = h_i,   h_i = psrc_i (rho_i - rho_prev_i) / 2,   dU_0 = dU_{N-1} = 0,
 *     a = (1 + delta/2)/2,  b = (1 - delta/2)/2  (the FP64 values the kernels use; delta = 0: the uniform grid, a = b = 1/2),
 * by the Thomas recurrence in __float128 (113-bit significand).  The system's condition grows like N^2 (~1e12 at 1048577 nodes): an FP64
 * solve carries errors of the size the tests look for, this one ~1e-22 relative.  Compiled by tests/poisson_increment_ref.py. */
#include <math.h>
#include <stdlib.h>

typedef __float128 q;

/* psrc_i = r_i 4 pi K_i as engine.cpp get_grid builds it (the same libm exp, the same operation order) */
void inc_psrc(int L, double delta, double max_r, double* psrc)
{
    const double kFourPi = 12.566370614359172;
    const int N = (1 << L) + 1;
    const int uniform = delta == 0.;
    const double h_uni = max_r / (double)(N - 1);
    const double rp = uniform ? 0. : max_r / (exp((double)(N - 1) * delta) - 1.);
    const double rp2d2 = rp * rp * (delta * delta);
    for (int i = 0; i < N; ++i) {
        const double ex = exp((double)i * delta);
        const double r = uniform ? (0. * (double)(N - 1 - i) + max_r * (double)i) / (double)(N - 1) : rp * (ex - 1.);
        const double K = uniform ? h_uni * h_uni : rp2d2 * exp((double)i * (2. * delta));
        psrc[i] = (i == 0 || i == N - 1) ? 0. : r * (kFourPi * K);
    }
}

/* dU[N] (rounded to FP64) of the system with right-hand side h[N] (h_0, h_{N-1} unused) */
void inc_solve_h(int N, double delta, const double* h, double* dU)
{
    const q a = (q)(0.5 * (1. + 0.5 * delta)), b = (q)(0.5 * (1. - 0.5 * delta));
    q* gam = (q*)malloc(sizeof(q) * (size_t)N);
    q* del = (q*)malloc(sizeof(q) * (size_t)N);
    gam[0] = 0; del[0] = 0;                                      /* dU_0 = 0 */
    for (int i = 1; i < N - 1; ++i) {
        const q w = 1 / (1 - a * gam[i - 1]);
        gam[i] = b * w;
        del[i] = w * ((q)h[i] + a * del[i - 1]);
    }
    q x = 0;                                                     /* dU_{N-1} = 0 */
    dU[N - 1] = 0.;
    for (int i = N - 2; i >= 1; --i) {
        x = gam[i] * x + del[i];
        dU[i] = (double)x;
    }
    dU[0] = 0.;
    free(gam); free(del);
}

/* n_dens densities: h_i = psrc_i (rho_i - rho_prev_i) / 2 formed in __float128 from the FP64 inputs; rho, rho_prev, dU [n_dens][N] */
void inc_solve(int L, double delta, double max_r, int n_dens, const double* rho, const double* rho_prev, double* dU)
{
    const int N = (1 << L) + 1;
    double* psrc = (double*)malloc(sizeof(double) * (size_t)N);
    inc_psrc(L, delta, max_r, psrc);
    const q a = (q)(0.5 * (1. + 0.5 * delta)), b = (q)(0.5 * (1. - 0.5 * delta));
    q* gam = (q*)malloc(sizeof(q) * (size_t)N);
    q* del = (q*)malloc(sizeof(q) * (size_t)N);
    for (int k = 0; k < n_dens; ++k) {
        const double* r = rho + (size_t)k * N;
        const double* p = rho_prev + (size_t)k * N;
        double* out = dU + (size_t)k * N;
        gam[0] = 0; del[0] = 0;
        for (int i = 1; i < N - 1; ++i) {
            const q hi = (q)psrc[i] * ((q)r[i] - (q)p[i]) / 2;
            const q w = 1 / (1 - a * gam[i - 1]);
            gam[i] = b * w;
            del[i] = w * (hi + a * del[i - 1]);
        }
        q x = 0;
        out[N - 1] = 0.;
        for (int i = N - 2; i >= 1; --i) {
            x = gam[i] * x + del[i];
            out[i] = (double)x;
        }
        out[0] = 0.;
    }
    free(psrc); free(gam); free(del);
}
