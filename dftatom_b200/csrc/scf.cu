// SCF state kernels: initial guess, orbital normalisation + density accumulation + mixing, VWN exchange-
// correlation + potential + the five energy integrals + the convergence test.  Everything stays on the device;
// the host only enqueues (engine.cpp).
//
// Replaces (reference DFTAtom/): DFTAtom.cpp:36-56 NormalizeNonUniform, :328-343 CalculateNonUniformDensity
// (mixing), :371-392 initial guess, :413-481 (LDA) and :937-1006 (LSDA) potential/energies/stop test,
// VWNExcCor.h:73-128 (LDA), :134-312 (LSDA), ExcCorBase.h:14-26, Integral.h:50-73 Simpson38.
#include "internal.h"
#include <cmath>

namespace dft {

// ---------------------------------------------------------------------------------------------------------
// VWN (Vosko-Wilk-Nusair) parametrisation, constants VWNExcCor.h:24-41
// ---------------------------------------------------------------------------------------------------------
struct VwnSet { double A, y0, b, c; };
__device__ __constant__ VwnSet kVwnP = { 0.0310907, -0.10498, 3.72744, 12.93532 };
__device__ __constant__ VwnSet kVwnF = { 0.01554535, -0.325, 7.06042, 18.0578 };
__device__ __constant__ VwnSet kVwnA = { -0.016886863940389628 /* -1/(6 pi^2) */, -0.0047584, 1.13107, 13.0045 };

struct VwnVal { double eps, deps; };

// eps: VWN eq. B.5 (VWNExcCor.h:43-50); deps: eq. B.6 (:52-55); y = sqrt(rs)
__device__ __forceinline__ VwnVal vwn_eval(double y, const VwnSet p)
{
    const double Y = y * (y + p.b) + p.c;
    const double Y0 = p.y0 * p.y0 + p.b * p.y0 + p.c;
    const double dy = y - p.y0;
    const double Q = sqrt(4. * p.c - p.b * p.b);
    const double at = atan(Q / (2. * y + p.b));
    VwnVal v;
    v.eps = p.A * (log(y * y / Y) + 2. * p.b / Q * at - p.b * p.y0 / Y0 * (log(dy * dy / Y) + 2. * (p.b + 2. * p.y0) / Q * at));
    v.deps = p.A * (p.c * dy - p.b * p.y0 * y) / (dy * Y);
    return v;
}

#define DFT_X1 0.6108870577108572        /* (3/(2 pi))^(2/3), VWNExcCor.h:75 */
#define DFT_CBRT2 1.2599210498948732
#define DFT_THREE_OVER_4PI 0.23873241463784300

struct XcLda { double vexc, edif; };
__device__ __forceinline__ XcLda xc_lda(double rho)
{   // VWNExcCor.h:73-128
    XcLda o; o.vexc = 0.; o.edif = 0.;
    if (rho < 1e-18) return o;
    const double third = 1. / 3.;
    const double rs = cbrt(3. / (kFourPi * rho));            // (the reference: pow(., 1/3) - equal to ~1e-16 relative, a fifth of the instructions)
    const VwnVal p = vwn_eval(sqrt(rs), kVwnP);
    o.vexc = -DFT_X1 / rs + p.eps - third * p.deps;
    o.edif = 0.25 * DFT_X1 / rs + third * p.deps;
    return o;
}

struct XcLsda { double va, vb, vexc, edif; };
__device__ __forceinline__ XcLsda xc_lsda(double roa, double rob)
{   // VWNExcCor.h:134-312, ExcCorBase.h:14-26
    XcLsda o; o.va = o.vb = o.vexc = o.edif = 0.;
    const double n = roa + rob;
    if (n < 1e-18) return o;
    const double third = 1. / 3.;
    const double rs = cbrt(3. / (kFourPi * n));
    const double rsa = cbrt(3. / (kFourPi * roa));
    const double rsb = cbrt(3. / (kFourPi * rob));
    const double exp_ = -DFT_X1 / rs;
    const double exdif = DFT_CBRT2 * exp_ - exp_;
    const double zeta = (roa - rob) / n;
    const double z3 = zeta * zeta * zeta, z4 = z3 * zeta;
    const double fdd = 4. / (9. * (DFT_CBRT2 - 1.));
    const double cp = cbrt(1. + zeta), cm = cbrt(1. - zeta);     // (1 +- zeta)^(1/3); ^(4/3) = x cbrt(x)
    const double fv = ((1. + zeta) * cp + (1. - zeta) * cm - 2.) / (2. * (DFT_CBRT2 - 1.));
    const double dfv = 2. / (3. * (DFT_CBRT2 - 1.)) * (cp - cm);
    const double y = sqrt(rs);
    const VwnVal P = vwn_eval(y, kVwnP), F = vwn_eval(y, kVwnF), A = vwn_eval(y, kVwnA);
    const double dfp = F.eps - P.eps;
    const double beta = fdd * dfp / A.eps - 1.;
    const double opbz4 = 1. + beta * z4;
    const double interp = fv / fdd * opbz4;
    const double betad = fdd / A.eps * (F.deps - P.deps - A.deps * dfp / A.eps);
    const double interpd = fv / fdd * z4 * betad;
    const double deriv = third * (P.deps + A.deps * interp + A.eps * interpd);
    const double dterm = A.eps / fdd * (4. * beta * z3 * fv + opbz4 * dfv);
    const double core = P.eps + A.eps * interp - deriv;
    o.va = -DFT_X1 * DFT_CBRT2 / rsa + core + (1. - zeta) * dterm;
    o.vb = -DFT_X1 * DFT_CBRT2 / rsb + core - (1. + zeta) * dterm;
    o.vexc = core + (exp_ + exdif * fv);
    const double expd = 0.25 * DFT_X1 / rs;
    o.edif = expd + (DFT_CBRT2 * expd - expd) * fv + deriv;
    return o;
}

__global__ void vwn_kernel(int n, const double* ra, const double* rb, double* va, double* vb, double* vexc, double* edif)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (rb) {
            const XcLsda x = xc_lsda(ra[i], rb[i]);
            va[i] = x.va; vb[i] = x.vb; vexc[i] = x.vexc; edif[i] = x.edif;
        } else {
            const XcLda x = xc_lda(ra[i]);
            vexc[i] = x.vexc; edif[i] = x.edif;
        }
    }
}

void launch_vwn(int n, const double* ra, const double* rb, double* va, double* vb, double* vexc, double* edif, cudaStream_t st)
{
    vwn_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, st>>>(n, ra, rb, va, vb, vexc, edif);
}

// Chachiyo's correlation with Dirac exchange (ExcCor.h:27-95; improved = the parameters of :20-25).  The reference reaches it from
// no option (comments only, DFTAtom.cpp:383,412,421): a component entry point, not part of the SCF path.
__global__ void chachiyo_kernel(int n, const double* rho, int improved, double* vexc, double* edif)
{
    const double a = (0.69314718055994530942 - 1.) / (2. * 3.14159265358979323846 * 3.14159265358979323846);      // (ln 2 - 1) / (2 pi^2)
    const double b = improved ? 21.7392245 : 20.4562557;
    const double X1 = pow(3. / (2. * 3.14159265358979323846), 2. / 3.);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double ro = rho[i];
        double v = 0., e = 0.;
        if (!(ro < 1E-18)) {
            const double rs = pow(3. / (kFourPi * ro), 1. / 3.);
            const double bprs = b / rs, bprs2 = bprs / rs;
            const double corr = a / (1. + bprs + bprs2) * (bprs + 2. * bprs2) * rs / 3.;
            v = -X1 / rs + a * log(1. + bprs + bprs / rs) - corr;
            e = 0.25 * X1 / rs + corr;
        }
        vexc[i] = v; edif[i] = e;
    }
}

void launch_chachiyo(int n, const double* rho, int improved, double* vexc, double* edif, cudaStream_t st)
{
    chachiyo_kernel<<<std::min((n + 255) / 256, 148 * 8), 256, 0, st>>>(n, rho, improved, vexc, edif);
}

// ---------------------------------------------------------------------------------------------------------
// block reductions
// ---------------------------------------------------------------------------------------------------------
template <int NV>
__device__ __forceinline__ void block_sum_n(double (&v)[NV], double* smem /* NV*32 doubles */)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
#pragma unroll
        for (int o = 16; o; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    }
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < NV; ++q) smem[q * 32 + w] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        double t = lane < nw ? smem[q * 32 + lane] : 0.;
#pragma unroll
        for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        v[q] = t;
    }
}

// Simpson38 weights of Integral.h:50-73 (times 3/8): ends 1, i%3==0 -> 2, else 3
__device__ __forceinline__ double simpson_w(int i, int n)
{
    const double w = (i == 0 || i == n - 1) ? 1. : ((i % 3 == 0) ? 2. : 3.);
    return w * 0.375;
}

__global__ void simpson38_kernel(double step, const double* v, int n, double* out)
{
    __shared__ double sm[32];
    const double* row = v + (size_t)blockIdx.x * n;
    double acc[1] = { 0. };
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc[0] = fma(simpson_w(i, n), row[i], acc[0]);
    block_sum_n<1>(acc, sm);
    if (threadIdx.x == 0) out[blockIdx.x] = acc[0] * step;
}

void launch_simpson38(double step, const double* v, int n, int n_rows, double* out, cudaStream_t st)
{
    simpson38_kernel<<<n_rows, 512, 0, st>>>(step, v, n, out);
}

// The other quadratures of Integral.h as block reductions (no call site in the reference's SCF; north_star names Romberg):
// rule 0 Trapezoid (Integral.h:11-23), 1 SimpsonOneThird (:25-48), 3 Boole (:75-104): one weighted sum; 4 Romberg (:106-155):
// the trapezoid refinements R(i,0) need the sum of the samples that are new at level i (stride numPoints >> (i-1), offset
// numPoints >> i) - one block reduction per level - then thread 0 runs the reference's extrapolation table and stop rule.
__device__ __forceinline__ double rule_weight(int rule, int i, int n)
{
    const bool end = (i == 0 || i == n - 1);
    if (rule == 0) return end ? 0.5 : 1.;
    if (rule == 1) return end ? 1. : ((i & 1) ? 4. : 2.);
    return end ? 7. : ((i & 1) ? 32. : ((i & 3) == 0 ? 14. : 12.));          // Boole
}

__global__ void __launch_bounds__(512) integrate_kernel(int rule, double step, const double* v, int n, double* out)
{
    __shared__ double sm[32];
    __shared__ double lsum[64];
    const double* row = v + (size_t)blockIdx.x * n;
    if (rule != 4) {
        double acc[1] = { 0. };
        for (int i = threadIdx.x; i < n; i += blockDim.x) acc[0] = fma(rule_weight(rule, i, n), row[i], acc[0]);
        block_sum_n<1>(acc, sm);
        const double coef = rule == 0 ? 1. : (rule == 1 ? 1. / 3. : 2. / 45.);
        if (threadIdx.x == 0) out[blockIdx.x] = acc[0] * step * coef;
        return;
    }
    const int numPoints = n - 1;
    int cnt = 0;
    for (int m = numPoints; m; m >>= 1) ++cnt;
    for (int i = 1; i < cnt; ++i) {
        const int oldStep = numPoints >> (i - 1), m = numPoints >> i;
        double acc[1] = { 0. };
        if (m > 0)
            for (long long j = m + (long long)threadIdx.x * oldStep; j < numPoints; j += (long long)blockDim.x * oldStep) acc[0] += row[j];
        block_sum_n<1>(acc, sm);
        if (threadIdx.x == 0) lsum[i] = acc[0];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double Rprev[24], Rcur[24];
        for (int q = 0; q < 24; ++q) { Rprev[q] = 0.; Rcur[q] = 0.; }
        double h = step * numPoints;
        Rprev[0] = 0.5 * h * (row[0] + row[numPoints]);
        double result = 0.;
        bool done = false;
        for (int i = 1; i < cnt && !done; ++i) {
            h *= 0.5;
            Rcur[0] = 0.5 * Rprev[0] + h * lsum[i];
            double nk = 1.;
            for (int q = 1; q <= i; ++q) {
                nk *= 4.;
                Rcur[q] = Rcur[q - 1] + (Rcur[q - 1] - Rprev[q - 1]) / (nk - 1.);
            }
            if (i >= 3 && fabs(Rcur[i] - Rprev[i - 1]) < 1e-18) { result = Rcur[i]; done = true; break; }
            for (int q = 0; q < 24; ++q) { const double t = Rcur[q]; Rcur[q] = Rprev[q]; Rprev[q] = t; }
        }
        out[blockIdx.x] = done ? result : Rprev[cnt - 1];
    }
}

void launch_integrate(int rule, double step, const double* v, int n, int n_rows, double* out, cudaStream_t st)
{
    if (rule == 2) simpson38_kernel<<<n_rows, 512, 0, st>>>(step, v, n, out);
    else integrate_kernel<<<n_rows, 512, 0, st>>>(rule, step, v, n, out);
}

// ---------------------------------------------------------------------------------------------------------
// SCF kernels, one CTA per atom
// ---------------------------------------------------------------------------------------------------------
constexpr int kAT = 512;

__global__ void __launch_bounds__(kAT) initial_density_kernel(GridDev g, ScfBuffers b)
{   // DFTAtom.cpp:371-376 / :876-884: uniform charge inside the sphere of radius MaxR
    const int a = blockIdx.x;
    const AtomDev at = b.atoms[a];
    const double volume = kFourPi / 3. * g.max_r * g.max_r * g.max_r;
    const int N = g.N;
    double* rt = b.rhot + (size_t)a * N;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        double tot = 0.;
        for (int s = 0; s < at.n_spin; ++s) {
            const double c = (i == 0) ? 0. : at.n_el[s] / volume;
            b.rho[(size_t)b.tab_of[2 * a + s] * N + i] = c;
            tot += c;
        }
        rt[i] = tot;
    }
}

void launch_initial_density(const GridDev& g, const ScfBuffers& b, cudaStream_t st)
{
    initial_density_kernel<<<b.n_atoms, kAT, 0, st>>>(g, b);
}

// LoopOverLevels' tail (normalise, accumulate occ u^2, Eel) + CalculateNonUniformDensity's mixing.
// psi holds the matched y_i of every orbital (inner part final, outer part already scaled).
// 1 / integral u^2 dr of every orbital, u_i = y_i e^{i δ/2}, dr = Rp δ e^{δ i} di  (DFTAtom.cpp:36-56); only needed after the
// validation-path match kernels, the production one (match_cta_kernel) returns it itself
__global__ void __launch_bounds__(256) orbital_norm_kernel(GridDev g, ScfBuffers b)
{
    __shared__ double red[8];
    const int o = blockIdx.x;
    if (b.astate[b.orbs[o].atom].done) return;
    const double* psi = b.psi + (size_t)o * g.N;
    double acc = 0.;
    for (int i = threadIdx.x; i < g.N; i += blockDim.x) {
        const double u = psi[i] * g.sqex[i];
        acc = fma(g.wjac[i], u * u, acc);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.;
        for (int v = 0; v < 8; ++v) tot += red[v];
        b.inv_norm[o] = 1. / tot;
    }
}

// New density and mixing (DFTAtom.cpp:558-559, :332-342).  grid = (atoms, node_chunks(N)): every CTA owns a contiguous range of
// nodes of one atom (the nodes are independent), so a handful of atoms still fills the GPU.
// node ranges per atom (gridDim.y): one per 512 nodes, 8..64 - both kernels are latency chains of loads per thread, and from the
// middle of a batch on only a few atoms are left, so short ranges on many SMs beat long ones on few
__host__ __device__ inline int node_chunks(int N) { const int c = (N + 511) / 512; return c < 8 ? 8 : (c > 64 ? 64 : c); }
constexpr int kDT = 256;
__global__ void __launch_bounds__(kDT) density_update_kernel(GridDev g, ScfBuffers b)
{
    DFT_PDL_WAIT();
    __shared__ double wgt[2 * DFTATOM_MAX_LEVELS];          // occupation / norm of every orbital
    const int a = blockIdx.x;
    AtomState& as = b.astate[a];
    if (as.done) return;
    const AtomDev at = b.atoms[a];
    const int N = g.N;
    for (int q = threadIdx.x; q < at.orb_count[0] + at.orb_count[1]; q += blockDim.x) {
        const int s = q >= at.orb_count[0];
        const int k = s ? q - at.orb_count[0] : q;
        const int o = at.orb_begin[s] + k;
        wgt[s * DFTATOM_MAX_LEVELS + k] = b.orbs[o].occ * b.inv_norm[o];
    }
    __syncthreads();
    const int per = (N + (int)gridDim.y - 1) / (int)gridDim.y;
    const int i0 = blockIdx.y * per, i1 = min(i0 + per, N);
    const double keep = b.adaptive_mixing ? as.mix : at.mixing, take = 1. - keep;
    double* rt = b.rhot + (size_t)a * N;
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double tot = 0.;
        const double sq = g.sqex[i];
        for (int s = 0; s < at.n_spin; ++s) {
            double acc = 0.;
            if (i < N - 1) {
                const double* p = b.psi + (size_t)at.orb_begin[s] * N + i;
                for (int k = 0; k < at.orb_count[s]; ++k) {
                    const double u = p[(size_t)k * N] * sq;
                    acc = fma(wgt[s * DFTATOM_MAX_LEVELS + k], u * u, acc);
                }
            }
            double* rho = b.rho + (size_t)b.tab_of[2 * a + s] * N;
            double r = rho[i];
            if (i >= 1) { r = keep * r + take * (acc * g.inv4pr2[i]); rho[i] = r; }
            tot += r;
        }
        if (at.n_spin == 2 && i >= 1) rt[i] = tot;     // DFTAtom.cpp:933-934 (LDA: rhot aliases rho)
        else if (at.n_spin == 1) rt[i] = tot;
    }
    // eigenvalues of this step into the record; electronic energy; reallyConverged
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        dftatom_step* rec = b.steps + (size_t)a * b.steps_stride + as.n_steps;
        double eel = 0.;
        int ok = 1;
        for (int s = 0; s < at.n_spin; ++s)
            for (int k = 0; k < at.orb_count[s]; ++k) {
                const int o = at.orb_begin[s] + k;
                const SearchState& st = b.ss[o];
                rec->E[s][k] = st.E;
                eel += b.orbs[o].occ * st.E;       // DFTAtom.cpp:561
                if (!st.converged) ok = 0;
            }
        rec->levels_converged = ok;
        rec->Ekin = eel;                                     // parked here until potential_energy_kernel
    }
}

void launch_orbital_norms(const GridDev& g, const ScfBuffers& b, cudaStream_t st)
{
    orbital_norm_kernel<<<b.n_orbs, 256, 0, st>>>(g, b);
}

void launch_density_update(const GridDev& g, const ScfBuffers& b, cudaStream_t st)
{
    launch_step_kernel(density_update_kernel, dim3(b.n_atoms, node_chunks(g.N)), dim3(kDT), 0, st, g, b);
}

// Potential from (U, rho), the five integrals, energies, stop test.  first != 0: only the initial potential.
// grid = (atoms, node_chunks(N)): every CTA owns a contiguous range of nodes; the partial sums of the five integrals go to
// b.epart, and the CTA that finishes last (per-atom ticket) adds them in chunk order - deterministic - and runs the stop test.
constexpr int kPT2 = 256;
// 3 CTAs per SM (80 registers, 256 B of spills): the kernel waits on the latency of log / atan / divisions of 2 nodes per thread - measured on the
// C3 sweep: 4.36 ms at 2 CTAs per SM (128 registers), 3.82 at 3, 3.60 at 4 (64 registers, 320 B of spills; no faster end to end)
#ifndef DFT_POT_MINB
#define DFT_POT_MINB 3
#endif
__global__ void __launch_bounds__(kPT2, DFT_POT_MINB) potential_energy_kernel(GridDev g, PoissonLevels lv, ScfBuffers b, int first)
{
    DFT_PDL_WAIT();
    __shared__ double sm[5 * 32];
    __shared__ int is_last;
    const int a = blockIdx.x;
    AtomState& as = b.astate[a];
    if (as.done) return;
    const AtomDev at = b.atoms[a];
    const int N = g.N;
    const double Z = (double)at.Z;
    const double* U = b.U + (size_t)a * b.ldU;               // U(r) = r V_H, written by the Poisson solve in natural node order
    const double* rt = b.rhot + (size_t)a * N;
    const int ta = b.tab_of[2 * a], tb = b.tab_of[2 * a + 1];
    const double q = g.delta * g.delta * 0.25;

    double e[5] = { 0., 0., 0., 0., 0. };   // nuclear, exccor, eexcDeriv, hartree, potentiale
    const int kPotChunks = (int)gridDim.y;
    const int per = (N + kPotChunks - 1) / kPotChunks;
    const int i0 = blockIdx.y * per, i1 = min(i0 + per, N);
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double Va = 0., Vb = 0.;
        if (i >= 1) {
            const double r = g.r[i];
            const double uc = (-Z + U[i]) / r;
            const double rho = rt[i];
            const double wj = g.wjac[i];                  // simpson weight x jacobian
            const double rd = r * rho * wj;
            const double r2d = r * rd;
            double vexc, edif, pot;
            if (at.n_spin == 2) {                          // DFTAtom.cpp:956-983
                const double ra = b.rho[(size_t)ta * N + i], rb = b.rho[(size_t)tb * N + i];
                const XcLsda x = xc_lsda(ra, rb);
                Va = uc + x.va; Vb = uc + x.vb;
                vexc = x.vexc; edif = x.edif;
                pot = r * r * wj * (ra * Va + rb * Vb);
            } else {                                       // DFTAtom.cpp:437-457
                const XcLda x = xc_lda(rho);
                Va = uc + x.vexc;
                vexc = x.vexc; edif = x.edif;
                pot = r2d * Va;
            }
            e[0] += Z * rd;
            e[1] = fma(r2d, vexc, e[1]);
            e[2] = fma(r2d, edif, e[2]);
            e[3] = fma(rd, U[i], e[3]);
            e[4] += pot;
        }
        b.vpot[(size_t)ta * N + i] = Va;
        b.atab[(size_t)ta * N + i] = (g.k2[i] * Va + q) * (1. / 12.);
        if (at.n_spin == 2) {
            b.vpot[(size_t)tb * N + i] = Vb;
            b.atab[(size_t)tb * N + i] = (g.k2[i] * Vb + q) * (1. / 12.);
        }
    }
    if (first) return;
    block_sum_n<5>(e, sm);
    if (threadIdx.x == 0) {
        double* part = b.epart + ((size_t)a * kPotChunks + blockIdx.y) * 5;
        for (int q = 0; q < 5; ++q) part[q] = e[q];
        __threadfence();
        const int ticket = atomicAdd(b.eticket + a, 1);
        is_last = (ticket == kPotChunks - 1);
        if (is_last) b.eticket[a] = 0;
    }
    __syncthreads();
    if (!is_last) return;
    // the CTA that finished last adds the partial sums in range order (deterministic): one thread per integral, loads from L2
    if (threadIdx.x < 5) {
        __threadfence();
        const double* part = b.epart + (size_t)a * kPotChunks * 5 + threadIdx.x;
        double t = 0.;
        for (int c = 0; c < kPotChunks; ++c) t += __ldcg(part + c * 5);
        sm[threadIdx.x] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 0; q < 5; ++q) e[q] = sm[q];
        dftatom_step* rec = b.steps + (size_t)a * b.steps_stride + as.n_steps;
        const double eel = rec->Ekin;                      // parked by density_update_kernel
        const double e_nuc = -kFourPi * e[0];              // DFTAtom.cpp:459-470
        const double e_dif = kFourPi * e[2];
        const double e_xc = kFourPi * e[1] + e_dif;
        const double e_har = -0.5 * kFourPi * e[3];
        const double e_pot = kFourPi * e[4];
        const double etot = eel + e_har + e_dif;
        rec->Etotal = etot; rec->Ekin = eel - e_pot; rec->Ecoul = -e_har; rec->Eenuc = e_nuc; rec->Exc = e_xc;
        const int ok = rec->levels_converged;
        int done = 0, status = DFTATOM_MAX_STEPS;
        const int crit = fabs((as.e_old - etot) / etot) < kTotalEnergyTol && ok && as.prev_ok;                                // :474
        rec->stop_criterion_met = crit;
        if (crit && !b.run_to_cap) { done = 1; status = DFTATOM_CONVERGED; }
        if (b.adaptive_mixing) {
            // Opt-in damping (default off: the reference's fixed linear mixing).  Linear mixing rho <- a rho + (1 - a) F(rho) sloshes with period 2
            // when the density response has an eigenvalue lambda < -(1 + a)/(1 - a) ~ -3 at a = 0.5 (nearly full nodeless 3d / 4f shells: Cu, Zn,
            // Ho .. Yb; the reference runs Er, Tm, Yb to its 100-step cap, SURVEY fact 5).  Detected as three energy changes of alternating sign
            // that decay by less than 2x per step; the cure is more of the old density: a <- (1 + a) / 2, at most three times, with a hold-off.
            const double d0 = etot - as.e_old;
            if (as.hold > 0) --as.hold;
            else if (as.n_steps >= 6 && as.n_raised < 3 && d0 * as.d1 < 0. && as.d1 * as.d2 < 0. && fabs(d0) > 0.5 * fabs(as.d1) && fabs(as.d1) > 0.5 * fabs(as.d2)) {
                as.mix = 0.5 * (1. + as.mix);
                as.hold = 4; as.n_raised += 1;
            }
            as.d2 = as.d1; as.d1 = d0;
        }
        as.e_old = etot;
        as.prev_ok = ok;
        as.n_steps += 1;
        if (!done && as.n_steps >= at.n_steps_max) { done = 1; status = DFTATOM_MAX_STEPS; }
        if (!done && !(fabs(etot) <= 1.7e308)) { done = 1; status = DFTATOM_NUMERIC_FAILURE; }
        if (done) { as.done = 1; as.status = status; atomicAdd(b.n_active, -1); atomicAdd(b.n_active + 1, -(at.orb_count[0] + at.orb_count[1])); }
    }
}

// Increment form of the warm-started Poisson solves.  A = the discrete operator is linear, so with U_prev the previous step's solution
//     U = U_prev + dU,   A dU = -(S - S_prev) = -r 4 pi K (rho - rho_prev),   dU = 0 on both boundaries.
// The plain warm start iterates on the residual S - A U_prev, whose three U terms cancel to ~1e-8 of their size: that cancellation is
// what puts every FP64 multigrid solve of U itself (the reference's included) on a rounding floor of ~1e-9 |U| that is a chaotic
// function of the input (tests/test_oracle.py::test_reference_poisson_floor_is_chaotic) and makes |dE/E| of consecutive SCF steps wander
// at 2e-11..1e-10.  Solved for the INCREMENT, every quantity in the solve is as small as the density change itself, its rounding is
// relative to dU, and the rounding-floor error of U stays frozen at what the last cold solve left: consecutive steps differ smoothly,
// and the stop test |dE/E| < 1e-11 (DFTAtom.cpp:474) fires when the energy has really stopped moving, not when the noise dips.
__global__ void __launch_bounds__(256) poisson_delta_prepare_kernel(int N, long long ld, const double* __restrict__ psrc, const double* __restrict__ rho,
                                                                    double* __restrict__ rho_prev, double* __restrict__ dS, double* __restrict__ dU,
                                                                    const int* skip, int skip_stride_bytes)
{
    const int k = blockIdx.y;
    if (skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(skip) + (size_t)k * skip_stride_bytes)) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double r = rho[(size_t)k * N + i];
    if (dS) {
        dS[(size_t)k * ld + i] = psrc[i] * (r - rho_prev[(size_t)k * N + i]);
        dU[(size_t)k * ld + i] = 0.;
    }
    rho_prev[(size_t)k * N + i] = r;
}
__global__ void __launch_bounds__(256) poisson_delta_apply_kernel(int N, long long ld, double* __restrict__ U, const double* __restrict__ dU,
                                                                  const int* skip, int skip_stride_bytes)
{
    const int k = blockIdx.y;
    if (skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(skip) + (size_t)k * skip_stride_bytes)) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) U[(size_t)k * ld + i] += dU[(size_t)k * ld + i];
}
void launch_poisson_delta_prepare(const GridDev& g, int n_dens, long long ld, const double* rho, double* rho_prev, double* dS, double* dU,
                                  const int* skip, int skip_stride_bytes, cudaStream_t st)
{
    poisson_delta_prepare_kernel<<<dim3((g.N + 255) / 256, n_dens), 256, 0, st>>>(g.N, ld, g.psrc, rho, rho_prev, dS, dU, skip, skip_stride_bytes);
}
void launch_poisson_delta_apply(const GridDev& g, int n_dens, long long ld, double* U, const double* dU, const int* skip, int skip_stride_bytes,
                                cudaStream_t st)
{
    poisson_delta_apply_kernel<<<dim3((g.N + 255) / 256, n_dens), 256, 0, st>>>(g.N, ld, U, dU, skip, skip_stride_bytes);
}

// Last node of the body of a phase of the SCF loop (one CUDA-graph WHILE node per phase = range of SCF steps [.., step_end), executed in
// order): the phase goes on while some atom is still iterating (n_active is kept up to date by potential_energy_kernel) and the next step
// is still its own; once no atom is left the later phases are switched off too.  step_first: the SCF step of the first graph iteration.
__global__ void scf_loop_condition_kernel(ScfLoopPhases ph, int phase, int step_first, int step_end, const int* n_active, unsigned long long* iterations)
{
    DFT_PDL_WAIT();
    const unsigned long long it = (*iterations += 1ULL);
    const bool active = *n_active > 0;
    cudaGraphSetConditional(ph.handle[phase], (active && (long long)step_first + (long long)it < (long long)step_end) ? 1u : 0u);
    if (!active) for (int q = phase + 1; q < ph.n; ++q) cudaGraphSetConditional(ph.handle[q], 0u);
}
void launch_scf_loop_condition(const ScfLoopPhases& ph, int phase, int step_first, int step_end, const int* n_active, unsigned long long* iterations, cudaStream_t st)
{
    launch_step_kernel(scf_loop_condition_kernel, dim3(1), dim3(1), 0, st, ph, phase, step_first, step_end, n_active, iterations);
}

__global__ void scale_unit_potential_kernel(int N, int ldU, const double* __restrict__ u1, const double* __restrict__ Q, double* __restrict__ U)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) U[(size_t)blockIdx.y * ldU + i] = Q[blockIdx.y] * u1[i];
}
void launch_scale_unit_potential(int N, int n_dens, int ldU, const double* u1, const double* Q, double* U, cudaStream_t st)
{
    scale_unit_potential_kernel<<<dim3((N + 255) / 256, n_dens), 256, 0, st>>>(N, ldU, u1, Q, U);
}

// last "Step:" record of every atom, compact (what dftatom_solve_batch downloads when the caller did not ask for the steps)
__global__ void gather_last_steps_kernel(ScfBuffers b, dftatom_step* out)
{
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= b.n_atoms) return;
    const int n = b.astate[a].n_steps;
    out[a] = b.steps[(size_t)a * b.steps_stride + (n > 0 ? n - 1 : 0)];
}
void launch_gather_last_steps(const ScfBuffers& b, dftatom_step* out, cudaStream_t st)
{
    gather_last_steps_kernel<<<(b.n_atoms + 127) / 128, 128, 0, st>>>(b, out);
}

void launch_potential_energy(const GridDev& g, const PoissonLevels& lv, const ScfBuffers& b, int first, cudaStream_t st)
{
    launch_step_kernel(potential_energy_kernel, dim3(b.n_atoms, node_chunks(g.N)), dim3(kPT2), 0, st, g, lv, b, first);
}

// The potential-and-energy step of a pseudo-atom (dftatom_solve_pseudo_batch): grid, per-atom ticket, fixed-order sum, stop test and
// adaptive mixing of potential_energy_kernel (the tail is repeated here so that kernel's code stays as it is).  Every channel row gets
// V_l,s = V_ion,l + U / r + V_xc,s and its a-table; the row tab_of[2 a + s] gets the screening U / r + V_xc,s (the radial export's v).
// The integrals: E_ion = sum occ <u|V_ion,l|u> and sum occ <u|V_l,s|u> over the orbitals in psi (occ x inv_norm x wjac x u^2), and
// the xc / Hartree integrals of the density as in the all-electron kernel.
// kCore (dftatom_solve_pseudo_batch_core; launched when some atom of the group has a core): an atom with p.pc_row[a] >= 0 takes V_xc,s of
// rho_s + rho_pc / 2 and the energies of the core-corrected definition - e[1] = sum_s rho_s v_xc,s, e[2] = rho eps_xc - e[1]'s integrand,
// e[5] = rho_pc eps_xc - so Etotal uses 4 pi (e[2] + e[5]); an atom without a core takes the operations and roundings of the kCore =
// false instance (its energy tail written out in explicit roundings below), so its records do not depend on the batch.
// Launch bounds: kCore = false keeps the plain (kPT2) bound (minimum 0 = none: the parent kernel's code, 128 registers); kCore = true
// asks for 1 CTA per SM, which lets ptxas use 188 registers without spills (at the 128 of 2 CTAs per SM it spills 68 B).
template <bool kCore>
__global__ void __launch_bounds__(kPT2, kCore ? 1 : 0) pseudo_potential_energy_kernel(GridDev g, ScfBuffers b, PseudoArgs p, int first)
{
    DFT_PDL_WAIT();
    constexpr int NE = kCore ? 6 : 5;
    __shared__ double sm[NE * 32];
    __shared__ double wgt[2 * DFTATOM_MAX_LEVELS];          // occupation / norm of every orbital
    __shared__ int orb_l[2 * DFTATOM_MAX_LEVELS];
    __shared__ int is_last;
    const int a = blockIdx.x;
    AtomState& as = b.astate[a];
    if (as.done) return;
    const AtomDev at = b.atoms[a];
    const PseudoAtomDev pd = p.atoms[a];
    const int N = g.N;
    const int n_orb = at.orb_count[0] + at.orb_count[1];
    if (!first)
        for (int q = threadIdx.x; q < n_orb; q += blockDim.x) {
            const int o = at.orb_begin[0] + q;          // the beta orbitals follow the alpha ones
            wgt[q] = b.orbs[o].occ * b.inv_norm[o];
            orb_l[q] = b.orbs[o].l;
        }
    __syncthreads();
    const double* U = b.U + (size_t)a * b.ldU;
    const double* rt = b.rhot + (size_t)a * N;
    const int ta = b.tab_of[2 * a], tb = b.tab_of[2 * a + 1];
    const double q = g.delta * g.delta * 0.25;
    const double* pc = nullptr;
    if (kCore) { const int pr = p.pc_row[a]; if (pr >= 0) pc = p.rho_pc + (size_t)pr * N; }

    double e[NE] = {};                      // E_ion, exccor, eexcDeriv, hartree, sum occ <u|V_l|u> (, core exccor)
    const int kPotChunks = (int)gridDim.y;
    const int per = (N + kPotChunks - 1) / kPotChunks;
    const int i0 = blockIdx.y * per, i1 = min(i0 + per, N);
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double S[2] = { 0., 0. };                           // screening per spin
        if (i >= 1) {
            const double r = g.r[i];
            const double vh = U[i] / r;
            const double rho = rt[i];
            const double wj = g.wjac[i];
            const double rd = r * rho * wj;
            const double r2d = r * rd;
            double vexc, edif;
            if (at.n_spin == 2) {
                const double ra = b.rho[(size_t)ta * N + i], rb = b.rho[(size_t)tb * N + i];
                double xa = ra, xb = rb;
                if (kCore && pc) { const double h = 0.5 * pc[i]; xa += h; xb += h; }
                const XcLsda x = xc_lsda(xa, xb);
                S[0] = vh + x.va; S[1] = vh + x.vb;
                vexc = x.vexc; edif = x.edif;
                if (kCore && pc) {          // sum_s rho_s v_xc,s is no longer rho vexc
                    const double sv = ra * x.va + rb * x.vb, rw = r * r * wj;
                    e[1] = fma(rw, sv, e[1]);
                    e[2] = fma(rw, rho * (vexc + edif) - sv, e[2]);
                }
            } else {
                const XcLda x = xc_lda((kCore && pc) ? rho + pc[i] : rho);
                S[0] = vh + x.vexc;
                vexc = x.vexc; edif = x.edif;
            }
            if (kCore && pc) {
                e[5] = fma(r * r * wj * pc[i], vexc + edif, e[5]);
                if (at.n_spin == 1) { e[1] = fma(r2d, vexc, e[1]); e[2] = fma(r2d, edif, e[2]); }
            } else {
                e[1] = fma(r2d, vexc, e[1]);
                e[2] = fma(r2d, edif, e[2]);
            }
            e[3] = fma(rd, U[i], e[3]);
            if (!first) {
                const double sq = g.sqex[i];
                for (int k = 0; k < n_orb; ++k) {
                    const int o = at.orb_begin[0] + k;
                    const double u = b.psi[(size_t)o * N + i] * sq;
                    const double w = wgt[k] * wj * u * u;
                    const double vi = p.v_ion[(size_t)pd.vrow[orb_l[k]] * N + i];
                    e[0] = fma(w, vi, e[0]);
                    e[4] = fma(w, vi + S[k >= at.orb_count[0]], e[4]);
                }
            }
        }
        for (int s = 0; s < at.n_spin; ++s) b.vpot[(size_t)(s ? tb : ta) * N + i] = S[s];
#pragma unroll
        for (int l = 0; l < 4; ++l) {
            if (pd.vrow[l] < 0) continue;
            const double vi = i >= 1 ? p.v_ion[(size_t)pd.vrow[l] * N + i] : 0.;
            for (int s = 0; s < at.n_spin; ++s) {
                const double V = i >= 1 ? vi + S[s] : 0.;
                const int t = pd.tab[s][l];
                b.vpot[(size_t)t * N + i] = V;
                b.atab[(size_t)t * N + i] = (g.k2[i] * V + q) * (1. / 12.);
            }
        }
    }
    if (first) return;
    block_sum_n<NE>(e, sm);
    if (threadIdx.x == 0) {
        double* part = b.epart + ((size_t)a * kPotChunks + blockIdx.y) * NE;
        for (int c = 0; c < NE; ++c) part[c] = e[c];
        __threadfence();
        const int ticket = atomicAdd(b.eticket + a, 1);
        is_last = (ticket == kPotChunks - 1);
        if (is_last) b.eticket[a] = 0;
    }
    __syncthreads();
    if (!is_last) return;
    if (threadIdx.x < NE) {
        __threadfence();
        const double* part = b.epart + (size_t)a * kPotChunks * NE + threadIdx.x;
        double t = 0.;
        for (int c = 0; c < kPotChunks; ++c) t += __ldcg(part + c * NE);
        sm[threadIdx.x] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int c = 0; c < NE; ++c) e[c] = sm[c];
        dftatom_step* rec = b.steps + (size_t)a * b.steps_stride + as.n_steps;
        const double eel = rec->Ekin;                      // parked by density_update_kernel
        const double e_har = -0.5 * kFourPi * e[3];
        double e_xc, etot;
        if constexpr (!kCore) {
            const double e_dif = kFourPi * e[2];
            e_xc = kFourPi * e[1] + e_dif;
            etot = eel + e_har + e_dif;
        } else if (pc) {
            const double e_dif = kFourPi * e[2] + kFourPi * e[5];
            e_xc = kFourPi * e[1] + e_dif;
            etot = eel + e_har + e_dif;
        } else {
            // an atom without a core: the roundings ptxas gives the kCore = false instance above (4 pi e[2] fused into both sums), written
            // out so that such an atom's records are bit-identical to dftatom_solve_pseudo_batch's
            e_xc = __fma_rn(e[2], kFourPi, __dmul_rn(kFourPi, e[1]));
            etot = __fma_rn(e[2], kFourPi, __dadd_rn(eel, e_har));
        }
        rec->Etotal = etot; rec->Ekin = eel - e[4]; rec->Ecoul = -e_har; rec->Eenuc = e[0]; rec->Exc = e_xc;
        const int ok = rec->levels_converged;
        int done = 0, status = DFTATOM_MAX_STEPS;
        const int crit = fabs((as.e_old - etot) / etot) < kTotalEnergyTol && ok && as.prev_ok;
        rec->stop_criterion_met = crit;
        if (crit && !b.run_to_cap) { done = 1; status = DFTATOM_CONVERGED; }
        if (b.adaptive_mixing) {                           // potential_energy_kernel's opt-in damping
            const double d0 = etot - as.e_old;
            if (as.hold > 0) --as.hold;
            else if (as.n_steps >= 6 && as.n_raised < 3 && d0 * as.d1 < 0. && as.d1 * as.d2 < 0. && fabs(d0) > 0.5 * fabs(as.d1) && fabs(as.d1) > 0.5 * fabs(as.d2)) {
                as.mix = 0.5 * (1. + as.mix);
                as.hold = 4; as.n_raised += 1;
            }
            as.d2 = as.d1; as.d1 = d0;
        }
        as.e_old = etot;
        as.prev_ok = ok;
        as.n_steps += 1;
        if (!done && as.n_steps >= at.n_steps_max) { done = 1; status = DFTATOM_MAX_STEPS; }
        if (!done && !(fabs(etot) <= 1.7e308)) { done = 1; status = DFTATOM_NUMERIC_FAILURE; }
        if (done) { as.done = 1; as.status = status; atomicAdd(b.n_active, -1); atomicAdd(b.n_active + 1, -n_orb); }
    }
}

void launch_pseudo_potential_energy(const GridDev& g, const ScfBuffers& b, const PseudoArgs& p, int first, cudaStream_t st)
{
    if (p.rho_pc) launch_step_kernel(pseudo_potential_energy_kernel<true>, dim3(b.n_atoms, node_chunks(g.N)), dim3(kPT2), 0, st, g, b, p, first);
    else launch_step_kernel(pseudo_potential_energy_kernel<false>, dim3(b.n_atoms, node_chunks(g.N)), dim3(kPT2), 0, st, g, b, p, first);
}

}  // namespace dft
