// Warm radial Poisson solves in increment form as ONE DIRECT SOLVE per density (grids of 2049 nodes and above).
//
// Replaces, for the warm solves of the SCF only (SCF step `warm_after` on), the V-cycles of PoissonSolver.h:155-159 / PoissonSolver.cpp:40-197.
// In increment form (scf.cu) a warm solve is the linear system of the FINEST level itself,
//     -a dU_{i-1} + dU_i - b dU_{i+1} = h_i,   h_i = r_i 4 pi K_i (rho_i - rho_prev_i) / 2,   dU_0 = dU_n = 0,   U += dU
// (the fixed point of the Gauss-Seidel sweep PoissonSolver.cpp:56-57 on level 0: a = (1 + delta/2)/2, b = (1 - delta/2)/2), which the
// reference's multigrid iterates towards and 7 V-cycles reach to ~1e-7 |dU|.  What has to look like the reference's solver is U itself:
// the rounding-floor bias of a plain FP64 multigrid solve, ~1e-9 |U| and worth ~1e-5 Ha at Z ~ 90 (DESIGN.md section 4.3), comes with
// the COLD full-multigrid solve of SCF step 0, which stays poisson_full_kernel.  The increments are 1e-2 .. 1e-9 of U: how their system
// is solved does not matter as long as it is solved, so it is solved exactly - Thomas algorithm, O(N), no iteration:
//     forward   delta_i = w_i (h_i + a delta_{i-1}),  w_i = 1 / (1 - a gamma_{i-1}),  gamma_i = b w_i        (pivots: a table of the grid)
//     backward  dU_i = gamma_i dU_{i+1} + delta_i.
// Both passes are first-order recurrences with multipliers -> 1 (every node sees every source), i.e. scans of affine maps that cannot be
// truncated: thread t owns NPT consecutive nodes (registers), runs its chunk with zero carry-in while accumulating the product of its
// multipliers, the 512 maps are combined by a warp scan + one scan over the 16 warp totals, and the carry is patched in.  One CTA per
// density; ~10 k cycles per solve against ~700 k for the 7 V-cycles of poisson_warm.cu.
#include "internal.h"
#include <algorithm>
#include <cmath>

namespace dft {
namespace {

constexpr int kDT = 512;             // threads per CTA
constexpr int kDStride = kDT + 1;    // owner-major stride of the staging array in shared memory

struct DShared {
    double wM[2][kDT / 32], wC[2][kDT / 32];      // per-warp totals of the affine maps, then their inclusive scan ([0] forward pass, [1] backward)
};
__shared__ DShared ds;
extern __shared__ double d_stage[];         // [NPT][513]: transposes between the coalesced natural order and the owners' rows

// inclusive scan of affine maps x -> M x + C over the threads of the CTA, in thread order (REVERSE: from the last thread down);
// returns the value entering this thread's chunk when `x_in` enters the first (REVERSE: last) thread's chunk
template <bool REVERSE>
__device__ __forceinline__ double block_carry(double M, double C, double x_in)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nw = kDT / 32;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double Mp = REVERSE ? __shfl_down_sync(full, M, o) : __shfl_up_sync(full, M, o);
        const double Cp = REVERSE ? __shfl_down_sync(full, C, o) : __shfl_up_sync(full, C, o);
        if (REVERSE ? (lane + o < 32) : (lane >= o)) { C = fma(M, Cp, C); M *= Mp; }
    }
    if (lane == (REVERSE ? 0 : 31)) { ds.wM[REVERSE][w] = M; ds.wC[REVERSE][w] = C; }
    // exclusive map of this lane inside its warp
    double Me = REVERSE ? __shfl_down_sync(full, M, 1) : __shfl_up_sync(full, M, 1);
    double Ce = REVERSE ? __shfl_down_sync(full, C, 1) : __shfl_up_sync(full, C, 1);
    if (lane == (REVERSE ? 31 : 0)) { Me = 1.; Ce = 0.; }
    __syncthreads();
    if (w == 0) {
        // the 16 warp maps: inclusive scan in warp order (REVERSE: from the last warp down), lanes >= 16 carry identities
        double Mw = lane < nw ? ds.wM[REVERSE][lane] : 1., Cw = lane < nw ? ds.wC[REVERSE][lane] : 0.;
#pragma unroll
        for (int o = 1; o < nw; o <<= 1) {
            const double Mp = REVERSE ? __shfl_down_sync(full, Mw, o) : __shfl_up_sync(full, Mw, o);
            const double Cp = REVERSE ? __shfl_down_sync(full, Cw, o) : __shfl_up_sync(full, Cw, o);
            if (REVERSE ? (lane + o < nw) : (lane >= o)) { Cw = fma(Mw, Cp, Cw); Mw *= Mp; }
        }
        if (lane < nw) { ds.wM[REVERSE][lane] = Mw; ds.wC[REVERSE][lane] = Cw; }
    }
    __syncthreads();
    // value entering this warp: the maps of the warps before it applied to x_in
    double xw = x_in;
    if (REVERSE ? (w + 1 < nw) : (w > 0)) { const int q = REVERSE ? w + 1 : w - 1; xw = fma(ds.wM[REVERSE][q], x_in, ds.wC[REVERSE][q]); }
    return fma(Me, xw, Ce);
}

template <int NPT>
__device__ __forceinline__ void direct_solve(const GridDev& g, const WarmPoissonArgs& a, int k)
{
    const int t = threadIdx.x;
    const int N = g.N, n = N - 1;                       // owned nodes 0 .. n-1 (node 0 and node n are the boundaries: dU = 0)
    const double* __restrict__ rho = a.rho + (size_t)k * a.rho_stride;
    double* __restrict__ rp = a.rho_prev + (size_t)k * a.rho_stride;
    double* __restrict__ U = a.U + (size_t)k * a.ldU;
    const double* __restrict__ W = g.coarse_direct;     // pivots w_i, owner-major: node i = t NPT + j at j 512 + t
    const double aa = 0.5 * (1. + 0.5 * g.delta), bb = 0.5 * (1. - 0.5 * g.delta);
    // import: h_i = r_i 4 pi K_i (rho_i - rho_prev_i) / 2 (coalesced) into the owners' rows; rho_prev = rho
    for (int i = t; i < N; i += kDT) {
        const double r = rho[i];
        const double base = rp[i];
        if (i < n) d_stage[(i % NPT) * kDStride + i / NPT] = (i >= 1) ? 0.5 * (g.psrc[i] * (r - base)) : 0.;
        rp[i] = r;
    }
    __syncthreads();
    double v[NPT];
    // forward elimination, local with zero carry-in; m = product of this thread's multipliers a w_i
    {
        double x = 0., m = 1.;
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const double w = W[j * kDT + t];
            const double aw = aa * w;
            x = fma(aw, x, w * d_stage[j * kDStride + t]);
            m *= aw;
            v[j] = x;
        }
        const double cin = block_carry<false>(m, x, 0.);      // delta at the node before this thread's first node
        double q = 1.;
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            q *= aa * W[j * kDT + t];
            v[j] = fma(q, cin, v[j]);
        }
    }
    // back substitution, local with zero carry-in from the right; m = product of this thread's multipliers gamma_i = b w_i
    {
        double y = 0., m = 1.;
#pragma unroll
        for (int j = NPT - 1; j >= 0; --j) {
            const double gm = bb * W[j * kDT + t];
            y = fma(gm, y, v[j]);
            m *= gm;
            v[j] = y;
        }
        const double pin = block_carry<true>(m, y, 0.);       // dU at the node after this thread's last node (dU_n = 0)
        double q = 1.;
#pragma unroll
        for (int j = NPT - 1; j >= 0; --j) {
            q *= bb * W[j * kDT + t];
            v[j] = fma(q, pin, v[j]);
        }
    }
    // export: U += dU (coalesced, through the owners' rows)
#pragma unroll
    for (int j = 0; j < NPT; ++j) d_stage[j * kDStride + t] = v[j];
    __syncthreads();
    for (int i = t; i < n; i += kDT) U[i] += d_stage[(i % NPT) * kDStride + i / NPT];
}

// Grids above 16385 nodes: the same two passes chunk by chunk (16384 nodes = 512 threads x 32), the carry of one chunk entering the next;
// delta of every chunk is parked in `scratch` (owner-major per chunk, coalesced) between the forward and the backward pass.
__device__ __forceinline__ void direct_solve_chunked(const GridDev& g, const WarmPoissonArgs& a, int k)
{
    constexpr int NPT = 32, CH = kDT * NPT;
    __shared__ double s_carry;
    const int t = threadIdx.x;
    const int N = g.N, n = N - 1, n_chunks = n / CH;
    const double* __restrict__ rho = a.rho + (size_t)k * a.rho_stride;
    double* __restrict__ rp = a.rho_prev + (size_t)k * a.rho_stride;
    double* __restrict__ U = a.U + (size_t)k * a.ldU;
    double* __restrict__ park = a.scratch + (size_t)k * a.scratch_stride;
    const double aa = 0.5 * (1. + 0.5 * g.delta), bb = 0.5 * (1. - 0.5 * g.delta);
    double v[NPT];
    if (t == 0) { s_carry = 0.; rp[n] = rho[n]; }
    for (int c = 0; c < n_chunks; ++c) {
        const double* __restrict__ W = g.coarse_direct + (size_t)c * CH;
        const int base = c * CH;
        __syncthreads();                                // (the previous chunk's rows and carry are done with)
        for (int q = t; q < CH; q += kDT) {
            const int i = base + q;
            const double r = rho[i];
            const double b0 = rp[i];
            d_stage[(q % NPT) * kDStride + q / NPT] = (i >= 1) ? 0.5 * (g.psrc[i] * (r - b0)) : 0.;
            rp[i] = r;
        }
        __syncthreads();
        const double d_in = s_carry;
        double x = 0., m = 1.;
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const double w = W[j * kDT + t];
            const double aw = aa * w;
            x = fma(aw, x, w * d_stage[j * kDStride + t]);
            m *= aw;
            v[j] = x;
        }
        const double cin = block_carry<false>(m, x, d_in);
        double qq = 1.;
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            qq *= aa * W[j * kDT + t];
            v[j] = fma(qq, cin, v[j]);
            park[(size_t)base + j * kDT + t] = v[j];
        }
        if (t == kDT - 1) s_carry = v[NPT - 1];          // (read by everybody after the barrier at the top of the next chunk)
    }
    __syncthreads();
    if (t == 0) s_carry = 0.;                            // dU_n = 0
    for (int c = n_chunks - 1; c >= 0; --c) {
        const double* __restrict__ W = g.coarse_direct + (size_t)c * CH;
        const int base = c * CH;
        __syncthreads();
        const double p_in = s_carry;
#pragma unroll
        for (int j = 0; j < NPT; ++j) v[j] = park[(size_t)base + j * kDT + t];
        double y = 0., m = 1.;
#pragma unroll
        for (int j = NPT - 1; j >= 0; --j) {
            const double gm = bb * W[j * kDT + t];
            y = fma(gm, y, v[j]);
            m *= gm;
            v[j] = y;
        }
        const double pin = block_carry<true>(m, y, p_in);
        double qq = 1.;
#pragma unroll
        for (int j = NPT - 1; j >= 0; --j) {
            qq *= bb * W[j * kDT + t];
            v[j] = fma(qq, pin, v[j]);
        }
#pragma unroll
        for (int j = 0; j < NPT; ++j) d_stage[j * kDStride + t] = v[j];
        __syncthreads();
        if (t == 0) s_carry = v[0];
        for (int q = t; q < CH; q += kDT) U[base + q] += d_stage[(q % NPT) * kDStride + q / NPT];
    }
}

}  // namespace

__global__ void __launch_bounds__(kDT, 1) poisson_direct_kernel(GridDev g, WarmPoissonArgs a)
{
    DFT_PDL_WAIT();
    const int k = blockIdx.x;
    if (a.skip && *reinterpret_cast<const int*>(reinterpret_cast<const char*>(a.skip) + (size_t)k * a.skip_stride_bytes)) return;
    switch (g.L) {
        case 14: direct_solve<32>(g, a, k); break;
        case 13: direct_solve<16>(g, a, k); break;
        case 12: direct_solve<8>(g, a, k); break;
        case 11: direct_solve<4>(g, a, k); break;
        default: direct_solve_chunked(g, a, k); break;  // 15 .. 20
    }
    if (threadIdx.x == 0 && a.work) atomicAdd(a.work, (unsigned long long)(2 * (g.N - 1)));      // (two elimination passes over the grid)
}

// pivots of the level-0 system of an L-level grid, owner-major for 512 owners (per chunk of 16384 nodes above 14 levels); built on the host once per
// grid (a dependent chain of n divisions: microseconds on a CPU core, milliseconds on one GPU thread); fma as the device code contracts it
void coarse_direct_host(int L, double delta, double* W)
{
    const int n = 1 << L;
    const int npt = n / kDT > 32 ? 32 : n / kDT, ch = kDT * npt;
    const double a = 0.5 * (1. + 0.5 * delta), b = 0.5 * (1. - 0.5 * delta);
    double gamma = 0.;
    for (int i = 0; i < n; ++i) {
        const double w = i ? 1. / std::fma(-a, gamma, 1.) : 0.;     // node 0: the left boundary (delta_0 = 0, gamma_0 = 0)
        gamma = b * w;
        const int c = i / ch, r = i % ch;
        W[(size_t)c * ch + (r % npt) * kDT + r / npt] = w;
    }
}

bool poisson_direct_supported(int L) { return L >= 11 && L <= 20; }
long long poisson_direct_table_doubles(int L) { return poisson_direct_supported(L) ? (1ll << L) : 0; }

static size_t direct_smem_bytes(int L) { return (size_t)std::min(32, (1 << L) / kDT) * kDStride * sizeof(double); }

int poisson_direct_init_device()
{
    DFT_CHECK(cudaFuncSetAttribute(poisson_direct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)direct_smem_bytes(14)));
    return 0;
}

// a: rho, rho_prev, U, skip (n_vcycles and coarse_tri are not used); g.coarse_direct must be set; above 14
// levels a.scratch (n_dens x scratch_stride doubles, scratch_stride >= N - 1) is required
void launch_poisson_direct(const GridDev& g, const WarmPoissonArgs& a, cudaStream_t st)
{
    launch_step_kernel(poisson_direct_kernel, dim3(a.n_dens), dim3(kDT), direct_smem_bytes(g.L), st, g, a);
}

}  // namespace dft
