/*
 * TEST INFRASTRUCTURE — NOT PART OF THE PRODUCT.
 *
 * The oracle's SCF for an electron configuration (orc_scf_config, dftatom_oracle_config.h): the drivers of dftatom_oracle.c
 * (orc_scf_ex, orc_scf_uniform) restated with double occupations, a start density of the configuration's electrons and the Hartree
 * boundary value Q = sum occ; the nucleus keeps Z.  Everything else - Numerov sweeps, level search, multigrid, VWN, quadrature - is
 * dftatom_oracle.c's own code, compiled into this library from that translation unit.  tests/test_config_host.py checks that the
 * Aufbau configuration reproduces orc_scf / orc_scf_uniform bit for bit.
 * Built by __graft_entry__.build() into oracle/libdftatom_oracle_config.so; loaded by tests/oracle_config_lib.py.
 */
#include "dftatom_oracle.c"
#include "dftatom_oracle_config.h"

/* SolvePoissonNonUniform, PoissonSolver.h:51-81, with boundary value U(max_r) = bc (the electron count) */
static void poisson_bc(int levels, double delta, double bc, double max_r, const double* rho, double* U,
                       int max_vcycles, double* vcycle_err, int* n_vcycles)
{
    mgrid* m = mg_new(levels, delta);
    const int n = m->size[0];
    double* S = m->src[0];
    const double rp0 = max_r / (exp((n - 1) * delta) - 1.);            /* FillRNonuniformR .cpp:212-223 */
    for (int i = 0; i < n; ++i) S[i] = rp0 * (exp(i * delta) - 1.);
    const double rp = max_r / (exp(((double)n - 1.) * delta) - 1.);    /* .h:65 */
    const double c = FOUR_PI * (rp * rp * (delta * delta));
    const double two_delta = 2. * delta;
    for (int i = 1; i < n - 1; ++i) S[i] *= c * exp(i * two_delta) * rho[i];
    m->lo_bc = 0; m->hi_bc = bc;
    const int k = mg_full_cycle(m, 1E-3, 1E-14, max_vcycles, vcycle_err);
    if (n_vcycles) *n_vcycles = k;
    memcpy(U, m->phi[0], sizeof(double) * (size_t)n);
    mg_free(m);
}

/* one orbital of the SCF: occupation as a double (a configuration's; the Aufbau's integers otherwise) */
typedef struct { int n0, l; double occ, E; } scf_level;

/* the records keep orc_level: occupation rounded to the nearest integer */
static void to_orc_levels(const scf_level* in, int n, orc_level* out)
{
    for (int k = 0; k < n; ++k) { out[k].n0 = in[k].n0; out[k].l = in[k].l; out[k].occ = (int)lround(in[k].occ); out[k].E = in[k].E; }
}

/* LoopOverLevels (:493-563) + the tail of CalculateNonUniformDensity (:332-342) for one spin channel */
static void cfg_channel_density(const double* V, int n, double delta, double max_r, double rp, double mixing,
                                 scf_level* lv, int n_lv, double Z, double* rho, double* acc, double* psi,
                                 double* e_el, int* all_converged)
{
    double bottom = -Z * Z - 1.;                                   /* :407 */
    memset(acc, 0, sizeof(double) * (size_t)n);
    for (int k = 0; k < n_lv; ++k) {
        int ok = 0;
        lv[k].E = orc_level_search(V, n, delta, max_r, lv[k].n0, lv[k].l, &bottom, &ok);
        if (!ok) *all_converged = 0;
        orc_numerov_match(V, n, delta, max_r, lv[k].l, lv[k].E, psi);      /* :545 */
        orc_normalize(psi, n, rp, delta);                                   /* :546 */
        for (int i = 0; i < n - 1; ++i) acc[i] += lv[k].occ * psi[i] * psi[i];   /* :558-559 */
        *e_el += lv[k].occ * lv[k].E;                                        /* :561 */
    }
    const double keep = mixing, take = 1. - mixing;
    for (int i = 1; i < n; ++i) {                                  /* :332-342 */
        const double r = rp * (exp(i * delta) - 1.);
        acc[i] /= FOUR_PI * r * r;
        rho[i] = keep * rho[i] + take * acc[i];
    }
}

/* The non-uniform SCF of the orbitals lv[spin][k] ((n, l) order) with n_el[spin] electrons: the start density is a uniform sphere of
 * n_el electrons per spin and the Hartree boundary value is Q = n_el[0] + n_el[1]; the nucleus keeps Z. */
static int scf_nonuniform(const orc_options* opt, scf_level lv[2][ORC_MAX_LEVELS], const int n_lv[2], const double n_el[2], orc_result* res,
                          orc_step_cb cb, void* user, int max_vcycles, double* V_out, double* rho_out)
{
    const int Z = opt->Z, lsda = opt->method != 0;
    const int n = orc_n_nodes(opt->levels);
    const double delta = opt->delta, max_r = opt->max_r;
    const double rp = max_r / (exp((n - 1) * delta) - 1.);
    const double Q = n_el[0] + n_el[1];
    const int n_spin = lsda ? 2 : 1;

    const size_t bytes = sizeof(double) * (size_t)n;
    double* rho_s[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* rho = lsda ? (double*)calloc(1, bytes) : rho_s[0];
    double* V[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* vxc_s[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* U = (double*)calloc(1, bytes), *vexc = (double*)calloc(1, bytes), *edif = (double*)calloc(1, bytes);
    double* acc = (double*)calloc(1, bytes), *psi = (double*)calloc(1, bytes);
    double* g_nuc = (double*)calloc(1, bytes), *g_xc = (double*)calloc(1, bytes), *g_dif = (double*)calloc(1, bytes);
    double* g_har = (double*)calloc(1, bytes), *g_pot = (double*)calloc(1, bytes);

    /* initial guess: uniform charge in the sphere, :371-376 / :876-884 */
    const double volume = FOUR_PI / 3. * max_r * max_r * max_r;
    if (lsda) {
        const double ca = n_el[0] / volume, cbeta = n_el[1] / volume;
        for (int i = 1; i < n; ++i) { rho_s[0][i] = ca; rho_s[1][i] = cbeta; rho[i] = ca + cbeta; }
    } else {
        const double c = Q / volume;
        for (int i = 1; i < n; ++i) rho[i] = c;
    }
    poisson_bc(opt->levels, delta, Q, max_r, rho, U, max_vcycles, NULL, NULL);
    if (lsda) orc_vwn_lsda(rho_s[0], rho_s[1], n, vxc_s[0], vxc_s[1], vexc, edif);
    else orc_vwn_lda(rho, n, vexc, edif);
    for (int i = 1; i < n; ++i) {                                  /* :387-392 / :895-904 */
        const double r = rp * (exp(i * delta) - 1.);
        if (lsda) { const double uc = (-Z + U[i]) / r; V[0][i] = uc + vxc_s[0][i]; V[1][i] = uc + vxc_s[1][i]; }
        else V[0][i] = (-Z + U[i]) / r + vexc[i];
    }

    const int max_steps = lsda ? 150 : 100;                        /* :396 / :908 */
    double e_old = 0;
    int prev_ok = 0;
    memset(res, 0, sizeof(*res));
    orc_step st;
    for (int sp = 0; sp < max_steps; ++sp) {
        memset(&st, 0, sizeof(st));
        st.step = sp;
        double e_el = 0;
        int ok = 1;
        for (int s = 0; s < n_spin; ++s)
            cfg_channel_density(V[s], n, delta, max_r, rp, opt->mixing, lv[s], n_lv[s], (double)Z, rho_s[s], acc, psi, &e_el, &ok);
        if (lsda) for (int i = 1; i < n; ++i) rho[i] = rho_s[0][i] + rho_s[1][i];   /* :933-934 */

        poisson_bc(opt->levels, delta, Q, max_r, rho, U, max_vcycles, NULL, NULL);
        if (lsda) orc_vwn_lsda(rho_s[0], rho_s[1], n, vxc_s[0], vxc_s[1], vexc, edif);
        else orc_vwn_lda(rho, n, vexc, edif);

        g_nuc[0] = g_xc[0] = g_dif[0] = g_har[0] = g_pot[0] = 0;
        V[0][0] = V[1][0] = 0;
        for (int i = 1; i < n; ++i) {
            const double ex = exp(delta * i);
            const double r = rp * (ex - 1.);
            const double jac = rp * delta * ex;
            if (!lsda) {                                           /* :437-457 */
                V[0][i] = (-Z + U[i]) / r + vexc[i];
                const double rd = r * rho[i] * jac;
                g_nuc[i] = Z * rd;
                const double r2d = r * r * rho[i] * jac;
                g_xc[i] = r2d * vexc[i];
                g_dif[i] = r2d * edif[i];
                g_har[i] = rd * U[i];
                g_pot[i] = r2d * V[0][i];
            } else {                                               /* :956-983 */
                const double uc = (-Z + U[i]) / r;
                V[0][i] = uc + vxc_s[0][i];
                V[1][i] = uc + vxc_s[1][i];
                const double rj = r * jac;
                const double rd = rj * rho[i];
                g_nuc[i] = Z * rd;
                const double r2j = r * rj;
                const double r2d = r2j * rho[i];
                g_xc[i] = r2d * vexc[i];
                g_dif[i] = r2d * edif[i];
                g_har[i] = rd * U[i];
                g_pot[i] = r2j * rho_s[0][i] * V[0][i] + r2j * rho_s[1][i] * V[1][i];
            }
        }
        const double e_nuc = -FOUR_PI * orc_simpson38(1, g_nuc, n);    /* :459-470 */
        double e_xc = FOUR_PI * orc_simpson38(1, g_xc, n);
        const double e_dif = FOUR_PI * orc_simpson38(1, g_dif, n);
        e_xc += e_dif;
        const double e_har = -2 * M_PI * orc_simpson38(1, g_har, n);
        const double e_pot = FOUR_PI * orc_simpson38(1, g_pot, n);
        st.Ekin = e_el - e_pot;
        st.Etotal = e_el + e_har + e_dif;
        st.Ecoul = -e_har;
        st.Eenuc = e_nuc;
        st.Exc = e_xc;
        st.level_search_converged = ok;
        for (int s = 0; s < n_spin; ++s) { st.n_levels[s] = n_lv[s]; to_orc_levels(lv[s], n_lv[s], st.lv[s]); }
        if (cb) cb(&st, user);
        res->n_steps = sp + 1;
        if (fabs((e_old - st.Etotal) / st.Etotal) < 1E-11 && ok && prev_ok) { res->finished = 1; break; }   /* :474-479 */
        e_old = st.Etotal;
        prev_ok = ok;
    }
    res->last = st;
    for (int s = 0; s < n_spin; ++s) {
        res->n_sorted[s] = n_lv[s];
        to_orc_levels(lv[s], n_lv[s], res->sorted[s]);
        sort_levels_by_energy(res->sorted[s], n_lv[s]);            /* :487 / :1012-1013 */
    }

    if (V_out) { memcpy(V_out, V[0], bytes); memcpy(V_out + n, V[1], bytes); }
    if (rho_out) { memcpy(rho_out, rho_s[0], bytes); memcpy(rho_out + n, rho_s[1], bytes); }
    free(rho_s[0]); free(rho_s[1]); if (lsda) free(rho);
    free(V[0]); free(V[1]); free(vxc_s[0]); free(vxc_s[1]); free(U); free(vexc); free(edif); free(acc); free(psi);
    free(g_nuc); free(g_xc); free(g_dif); free(g_har); free(g_pot);
    return 0;
}

/* SolvePoissonUniform, PoissonSolver.h:20-49 (constructor with dGrid = 0: no first-derivative term), boundary value bc */
static void poisson_uniform_bc(int levels, double bc, double max_r, const double* rho, double* U, int max_vcycles)
{
    mgrid* m = mg_new(levels, 0.);
    const int n = m->size[0];
    double* S = m->src[0];
    const size_t N = (size_t)n - 1;
    for (size_t i = 0; i < (size_t)n; ++i) S[i] = (0. * (N - i) + max_r * i) / N;      /* FillR, PoissonSolver.cpp:199-209 */
    const double delta = S[1] - S[0];
    const double c = (delta * delta) * FOUR_PI;
    for (int i = 0; i < n; ++i) S[i] *= c * rho[i];
    m->lo_bc = 0; m->hi_bc = bc;
    mg_full_cycle(m, 1E-3, 1E-14, max_vcycles, NULL);
    memcpy(U, m->phi[0], sizeof(double) * (size_t)n);
    mg_free(m);
}

/* LoopOverLevels :213-284 (with LocateInterval :287-325 and NormalizeUniform :21-32) + the mixing loop of the drivers */
static void cfg_channel_density_uniform(const double* V, int n, double max_r, double h, double mixing, scf_level* lv, int n_lv, double Z,
                                         double* rho, double* acc, double* psi, double* sq, double* e_el, int* all_converged)
{
    const double tol = 1E-12;
    const long n_steps = n - 1;
    double bottom = -Z * Z - 1.;
    memset(acc, 0, sizeof(double) * (size_t)n);
    for (int k = 0; k < n_lv; ++k) {
        const int l = lv[k].l, want = lv[k].n0 - l;
        double top = 50;
        double hi = top, lo = bottom;                               /* LocateInterval */
        while (hi - lo > tol) {
            const double E = (hi + lo) / 2;
            if (orc_u_count_nodes(V, max_r, l, E, n_steps, want) > want) hi = E; else lo = E;
        }
        top = hi;
        lo = bottom;
        while (hi - lo > tol) {
            const double E = (hi + lo) / 2;
            if (orc_u_count_nodes(V, max_r, l, E, n_steps, want) < want) lo = E; else hi = E;
        }
        bottom = hi;
        double y0 = orc_u_y0(V, max_r, l, bottom, n_steps);         /* :234-254 */
        const int sign_bottom = y0 > 0;
        int ok = 0;
        double E = bottom;
        for (int it = 0; it < 500; ++it) {
            E = (top + bottom) / 2;
            y0 = orc_u_y0(V, max_r, l, E, n_steps);
            if ((y0 > 0) == sign_bottom) bottom = E; else top = E;
            const double a = fabs(y0);
            if (top - bottom < tol && !isnan(a) && a < 1E15) { ok = 1; break; }
        }
        lv[k].E = bottom;                                           /* :255 */
        if (!ok) *all_converged = 0;
        bottom = lv[k].E - 3;                                       /* :262 */
        orc_u_match(V, max_r, l, lv[k].E, n_steps, psi);            /* :266 */
        for (int i = 0; i < n; ++i) sq[i] = psi[i] * psi[i];        /* NormalizeUniform */
        const double unorm = 1. / sqrt(orc_simpson38(h, sq, n));
        for (int i = 0; i < n; ++i) psi[i] *= unorm;
        for (int i = 0; i < n - 1; ++i) acc[i] += lv[k].occ * psi[i] * psi[i];    /* :279-280 */
        *e_el += lv[k].occ * lv[k].E;
    }
    const double keep = mixing, take = 1. - mixing;
    for (int i = 1; i < n; ++i) {                                   /* :127-137 / :713-718 */
        const double position = i * h;
        acc[i] /= FOUR_PI * position * position;
        rho[i] = keep * rho[i] + take * acc[i];
    }
}

/* the uniform-grid SCF of the orbitals lv with n_el electrons per spin (as scf_nonuniform); opt->method 2 = LDA, 3 = LSDA */
static int scf_uniform(const orc_options* opt, scf_level lv[2][ORC_MAX_LEVELS], const int n_lv[2], const double n_el[2], orc_result* res,
                       orc_step_cb cb, void* user, int max_vcycles, double* V_out, double* rho_out)
{
    const int Z = opt->Z, lsda = opt->method == 3;
    const int n = orc_n_nodes(opt->levels);
    const double max_r = opt->max_r;
    const double h = max_r / (n - 1);
    const double Q = n_el[0] + n_el[1];
    const int n_spin = lsda ? 2 : 1;

    const size_t bytes = sizeof(double) * (size_t)n;
    double* rho_s[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* rho = lsda ? (double*)calloc(1, bytes) : rho_s[0];
    double* V[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* vxc_s[2] = { (double*)calloc(1, bytes), (double*)calloc(1, bytes) };
    double* U = (double*)calloc(1, bytes), *vexc = (double*)calloc(1, bytes), *edif = (double*)calloc(1, bytes);
    double* acc = (double*)calloc(1, bytes), *psi = (double*)calloc(1, bytes), *sq = (double*)calloc(1, bytes);
    double* g_nuc = (double*)calloc(1, bytes), *g_xc = (double*)calloc(1, bytes), *g_dif = (double*)calloc(1, bytes);
    double* g_har = (double*)calloc(1, bytes), *g_pot = (double*)calloc(1, bytes);

    const double volume = 4. / 3. * M_PI * max_r * max_r * max_r;   /* :83 / :671 */
    if (lsda) {
        const double ca = n_el[0] / volume, cbeta = n_el[1] / volume;
        for (int i = 1; i < n; ++i) { rho_s[0][i] = ca; rho_s[1][i] = cbeta; rho[i] = ca + cbeta; }
    } else {
        const double c = Q / volume;
        for (int i = 1; i < n; ++i) rho[i] = c;
    }
    poisson_uniform_bc(opt->levels, Q, max_r, rho, U, max_vcycles);
    if (lsda) orc_vwn_lsda(rho_s[0], rho_s[1], n, vxc_s[0], vxc_s[1], vexc, edif);
    else orc_vwn_lda(rho, n, vexc, edif);
    for (int i = 1; i < n; ++i) {                                   /* :97-102 / :688-695 */
        const double pos = h * i;
        if (lsda) { const double uc = (-Z + U[i]) / pos; V[0][i] = uc + vxc_s[0][i]; V[1][i] = uc + vxc_s[1][i]; }
        else V[0][i] = (-Z + U[i]) / pos + vexc[i];
    }

    const int max_steps = lsda ? 150 : 100;                         /* :106 / :699 */
    double e_old = 0;
    int prev_ok = 0;
    memset(res, 0, sizeof(*res));
    orc_step st;
    for (int sp = 0; sp < max_steps; ++sp) {
        memset(&st, 0, sizeof(st));
        st.step = sp;
        double e_el = 0;
        int ok = 1;
        for (int s = 0; s < n_spin; ++s)
            cfg_channel_density_uniform(V[s], n, max_r, h, opt->mixing, lv[s], n_lv[s], (double)Z, rho_s[s], acc, psi, sq, &e_el, &ok);
        if (lsda) for (int i = 1; i < n; ++i) rho[i] = rho_s[0][i] + rho_s[1][i];

        poisson_uniform_bc(opt->levels, Q, max_r, rho, U, max_vcycles);
        if (lsda) orc_vwn_lsda(rho_s[0], rho_s[1], n, vxc_s[0], vxc_s[1], vexc, edif);
        else orc_vwn_lda(rho, n, vexc, edif);

        g_nuc[0] = g_xc[0] = g_dif[0] = g_har[0] = g_pot[0] = 0;
        V[0][0] = V[1][0] = 0;
        for (int i = 1; i < n; ++i) {
            const double position = i * h;
            if (!lsda) {                                            /* :160-180 */
                V[0][i] = (-Z + U[i]) / position + vexc[i];
                const double pd = position * rho[i];
                g_nuc[i] = Z * pd;
                const double p2d = position * position * rho[i];
                g_xc[i] = p2d * vexc[i];
                g_dif[i] = p2d * edif[i];
                g_har[i] = pd * U[i];
                g_pot[i] = p2d * V[0][i];
            } else {                                                /* :786-806 */
                const double uc = (-Z + U[i]) / position;
                V[0][i] = uc + vxc_s[0][i];
                V[1][i] = uc + vxc_s[1][i];
                const double pd = position * rho[i];
                g_nuc[i] = Z * pd;
                const double p2 = position * position;
                const double p2d = p2 * rho[i];
                g_xc[i] = p2d * vexc[i];
                g_dif[i] = p2d * edif[i];
                g_har[i] = pd * U[i];
                g_pot[i] = p2 * (rho_s[0][i] * V[0][i] + rho_s[1][i] * V[1][i]);
            }
        }
        const double e_nuc = -FOUR_PI * orc_simpson38(h, g_nuc, n);     /* :182-194 */
        double e_xc = 4 * M_PI * orc_simpson38(h, g_xc, n);
        const double e_dif = FOUR_PI * orc_simpson38(h, g_dif, n);
        e_xc += e_dif;
        const double e_har = -2 * M_PI * orc_simpson38(h, g_har, n);
        const double e_pot = FOUR_PI * orc_simpson38(h, g_pot, n);
        st.Ekin = e_el - e_pot;
        st.Etotal = e_el + e_har + e_dif;
        st.Ecoul = -e_har;
        st.Eenuc = e_nuc;
        st.Exc = e_xc;
        st.level_search_converged = ok;
        for (int s = 0; s < n_spin; ++s) { st.n_levels[s] = n_lv[s]; to_orc_levels(lv[s], n_lv[s], st.lv[s]); }
        if (cb) cb(&st, user);
        res->n_steps = sp + 1;
        if (fabs((e_old - st.Etotal) / st.Etotal) < 1E-11 && ok && prev_ok) { res->finished = 1; break; }   /* :198-203 */
        e_old = st.Etotal;
        prev_ok = ok;
    }
    res->last = st;
    for (int s = 0; s < n_spin; ++s) {
        res->n_sorted[s] = n_lv[s];
        to_orc_levels(lv[s], n_lv[s], res->sorted[s]);
        sort_levels_by_energy(res->sorted[s], n_lv[s]);
    }
    if (V_out) { memcpy(V_out, V[0], bytes); memcpy(V_out + n, V[1], bytes); }
    if (rho_out) { memcpy(rho_out, rho_s[0], bytes); memcpy(rho_out + n, rho_s[1], bytes); }
    free(rho_s[0]); free(rho_s[1]); if (lsda) free(rho);
    free(V[0]); free(V[1]); free(vxc_s[0]); free(vxc_s[1]); free(U); free(vexc); free(edif); free(acc); free(psi); free(sq);
    free(g_nuc); free(g_xc); free(g_dif); free(g_har); free(g_pot);
    return 0;
}

int orc_scf_config(const orc_options* opt, const orc_config* cfg, orc_result* res, orc_step_cb cb, void* user, int max_vcycles,
                   double* V_out, double* rho_out)
{
    const int lsda = opt->method & 1;
    scf_level lv[2][ORC_MAX_LEVELS];
    int n_lv[2] = { 0, 0 };
    double n_el[2] = { 0, 0 };
    if (!cfg || cfg->n_orbitals < 0 || cfg->n_orbitals > 2 * ORC_MAX_LEVELS || opt->method < 0 || opt->method > 3) return -1;
    for (int s = 0; s < 2; ++s) {
        for (int k = 0; k < cfg->n_orbitals; ++k) {
            const orc_orbital* o = &cfg->orb[k];
            if (o->spin != s) continue;
            if (o->n < 1 || o->l < 0 || o->l >= o->n || (s == 1 && !lsda) || n_lv[s] == ORC_MAX_LEVELS) return -1;
            int j = n_lv[s]++;                                   /* insertion into (n, l) order */
            while (j > 0 && (lv[s][j - 1].n0 > o->n - 1 || (lv[s][j - 1].n0 == o->n - 1 && lv[s][j - 1].l > o->l))) { lv[s][j] = lv[s][j - 1]; --j; }
            lv[s][j].n0 = o->n - 1; lv[s][j].l = o->l; lv[s][j].occ = o->occ; lv[s][j].E = 0;
        }
        for (int k = 0; k < n_lv[s]; ++k) n_el[s] += lv[s][k].occ;
    }
    if (n_lv[0] == 0) return -1;
    if (opt->method >= 2) return scf_uniform(opt, lv, n_lv, n_el, res, cb, user, max_vcycles, V_out, rho_out);
    return scf_nonuniform(opt, lv, n_lv, n_el, res, cb, user, max_vcycles, V_out, rho_out);
}
