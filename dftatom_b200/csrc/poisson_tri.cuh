// Exact solve of the 1024-node correction level of the radial Poisson V-cycle by one warp (poisson_warm.cu).
//
// The reference's V-cycle (PoissonSolver.h:155-159, PoissonSolver.cpp:162-197) visits, below the 1024-node level, the levels of 512 .. 2
// nodes with 3 + 3 Gauss-Seidel sweeps each: ~60 dependent sweeps of ~1100 cycles for a few hundred nodes - a quarter to a third of a
// solve on the GPU, with all but one warp idle.  That sub-cycle is an approximate solve of the level's own equation
//     -a Phi_{i-1} + Phi_i - b Phi_{i+1} = S_i / 2,   Phi_0 = Phi_n = 0            (the fixed point of PoissonSolver.cpp:56-57 on that level)
// entered with Phi = 0.  Here it is replaced by the EXACT solution of that equation (Thomas algorithm; the pivots depend on the grid only
// and come from a table): a coarse-grid correction that is at least as good, so the V-cycle converges to the same level-0 fixed point in
// no more cycles; the sweeps, restrictions and prolongations of the levels >= 2048 nodes - where the rounding behaviour of the solve is
// decided (DESIGN.md section 4.3) - are untouched.  Both elimination passes are first-order recurrences with NON-contractive multipliers
// (that is what makes the solve exact: every node sees every source), so they are run as 32 nodes per lane + a full warp scan of the
// affine maps + a patch with tabulated prefix / suffix products: ~2 k cycles instead of ~30 k.
#pragma once
#include <cuda_runtime.h>

namespace dft {

constexpr int kTriN = 1024;                     // owned nodes of the level (node 0 = left boundary, node 1024 = right boundary)
constexpr int kTriTableDoubles = 3 * kTriN;     // W, ML, GL, each in the layout [k * 32 + lane] for node i = 32 lane + k

// table for level spacing d (= delta 2^l of that level): one thread
//   w_0 = 0, w_i = 1 / (1 - a gamma_{i-1}), gamma_i = b w_i                               (pivots of the forward elimination)
//   ML_i = prod_{j = 32 lane .. i} a w_j,  GL_i = prod_{j = i .. 32 lane + 31} b w_j      (local prefix / suffix products of the multipliers)
inline __host__ __device__ void tri_build_table(double d, double* T)
{
    const double a = 0.5 * (1. + 0.5 * d), b = 0.5 * (1. - 0.5 * d);
    double* W = T; double* ML = T + kTriN; double* GL = T + 2 * kTriN;
    double gamma = 0.;
    for (int i = 0; i < kTriN; ++i) {
        const double w = i ? 1. / fma(-a, gamma, 1.) : 0.;
        gamma = b * w;
        W[(i & 31) * 32 + (i >> 5)] = w;
    }
    for (int lane = 0; lane < 32; ++lane) {
        double p = 1.;
        for (int k = 0; k < 32; ++k) { p *= a * W[k * 32 + lane]; ML[k * 32 + lane] = p; }
        p = 1.;
        for (int k = 31; k >= 0; --k) { p *= b * W[k * 32 + lane]; GL[k * 32 + lane] = p; }
    }
}

// warp-collective: hload(i) = S_i / 2, pstore(i, Phi_i) for the nodes i = 32 lane .. 32 lane + 31; T: the table (shared memory)
template <class HL, class PS>
__device__ __forceinline__ void tri_solve_warp(const double* __restrict__ T, double a, double b, HL hload, PS pstore)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const double* W = T + lane; const double* ML = T + kTriN + lane; const double* GL = T + 2 * kTriN + lane;
    double v[32];
    // forward elimination: delta_i = w_i (h_i + a delta_{i-1}), local with zero carry-in
    double x = 0.;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        const double w = W[k * 32];
        x = fma(a * w, x, w * hload(lane * 32 + k));
        v[k] = x;
    }
    {
        double M = ML[31 * 32], C = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double Mp = __shfl_up_sync(full, M, o), Cp = __shfl_up_sync(full, C, o);
            if (lane >= o) { C = fma(M, Cp, C); M *= Mp; }
        }
        double din = __shfl_up_sync(full, C, 1);
        if (lane == 0) din = 0.;
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = fma(ML[k * 32], din, v[k]);
    }
    // back substitution: Phi_i = gamma_i Phi_{i+1} + delta_i, local with zero carry-in from the right
    double y = 0.;
#pragma unroll
    for (int k = 31; k >= 0; --k) {
        y = fma(b * W[k * 32], y, v[k]);
        v[k] = y;
    }
    {
        double G = GL[0], C = y;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double Gp = __shfl_down_sync(full, G, o), Cp = __shfl_down_sync(full, C, o);
            if (lane + o < 32) { C = fma(G, Cp, C); G *= Gp; }
        }
        double pin = __shfl_down_sync(full, C, 1);
        if (lane == 31) pin = 0.;                   // Phi_n = 0: a correction level
#pragma unroll
        for (int k = 0; k < 32; ++k) pstore(lane * 32 + k, fma(GL[k * 32], pin, v[k]));
    }
}

}  // namespace dft
