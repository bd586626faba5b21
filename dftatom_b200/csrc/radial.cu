// Export of the converged radial state of the SCF (dftatom_solve_batch_radial) and the moment reduction of caller-supplied orbitals
// (dftatom_radial_moments).  Runs after the SCF loop on the group's stream; reads the SCF arrays, never writes them.
//
// Both kernels have the grid shape of density_update_kernel (scf.cu): one CTA per (row, node range).  Every CTA writes its nodes to
// the packed staging buffer and its partial sums to a per-range slot; the CTA that arrives last at the row's ticket adds the slots in
// range order (the epart / eticket pattern of potential_energy_kernel), so the moments do not depend on the order the CTAs ran in.
#include "internal.h"

namespace dft {

constexpr int kRT = 256;
// node ranges per row: the same count density_update_kernel uses (one per 512 nodes, 8..64)
static inline int radial_chunks(int N) { const int c = (N + 511) / 512; return c < 8 ? 8 : (c > 64 ? 64 : c); }

template <int NV>
__device__ __forceinline__ void radial_block_sum(double (&v)[NV], double* smem /* NV * 32 */)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int q = 0; q < NV; ++q)
#pragma unroll
        for (int o = 16; o; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < NV; ++q) smem[q * 32 + w] = v[q];
    __syncthreads();
    if (threadIdx.x == 0)
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            double t = 0.;
            for (int k = 0; k < nw; ++k) t += smem[q * 32 + k];
            v[q] = t;
        }
}

// Partial sums of one CTA into its slot; returns true in the CTA that arrived last, whose thread 0 then holds the row's totals in v
template <int NV>
__device__ __forceinline__ bool radial_finish(double (&v)[NV], double* part /* [gridDim.y][NV] of this row */, int* ticket, double* smem)
{
    __shared__ int is_last;
    radial_block_sum<NV>(v, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int q = 0; q < NV; ++q) part[blockIdx.y * NV + q] = v[q];
        __threadfence();
        is_last = atomicAdd(ticket, 1) == (int)gridDim.y - 1;
    }
    __syncthreads();
    if (!is_last) return false;
    if (threadIdx.x == 0) {
        __threadfence();
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            double t = 0.;
            for (int c = 0; c < (int)gridDim.y; ++c) t += __ldcg(part + c * NV + q);
            v[q] = t;
        }
    }
    return true;
}

// One row per orbital.  from_scf: u_i = sign * psi_i * sqex_i * sqrt(inv_norm) - the u whose square density_update_kernel accumulates -
// with the sign that makes u positive at the first node away from the nucleus where it is non-zero; otherwise u = src as given.
// Moments with the Simpson38-weighted jacobian of the energies: <1/r> (node 0, r = 0, left out), <r>, <r^2>.
__global__ void __launch_bounds__(kRT) radial_orbitals_kernel(GridDev g, const double* __restrict__ src, const double* __restrict__ inv_norm,
                                                              int from_scf, double* __restrict__ u_out, double* __restrict__ moments,
                                                              double* __restrict__ part, int* __restrict__ ticket)
{
    __shared__ double smem[3 * 32];
    __shared__ double scale;
    const int o = blockIdx.x, N = g.N;
    const double* p = src + (size_t)o * N;
    if (threadIdx.x == 0) {
        double s = 1.;
        if (from_scf) {
            int i = 1;
            while (i < N - 1 && p[i] == 0.) ++i;
            s = (p[i] < 0. ? -1. : 1.) * sqrt(inv_norm[o]);
        }
        scale = s;
    }
    __syncthreads();
    const double sc = scale;
    const int per = (N + (int)gridDim.y - 1) / (int)gridDim.y;
    const int i0 = blockIdx.y * per, i1 = min(i0 + per, N);
    double* u = u_out ? u_out + (size_t)o * N : nullptr;
    double m[3] = { 0., 0., 0. };
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double v = p[i];
        if (from_scf) v *= g.sqex[i] * sc;
        if (u) u[i] = v;
        const double r = g.r[i], w = g.wjac[i] * v * v;
        if (i > 0) m[0] = fma(w, 1. / r, m[0]);
        m[1] = fma(w, r, m[1]);
        m[2] = fma(w, r * r, m[2]);
    }
    if (radial_finish<3>(m, part + (size_t)o * gridDim.y * 3, ticket + o, smem) && threadIdx.x == 0) {
        for (int q = 0; q < 3; ++q) moments[(size_t)o * DFTATOM_N_MOMENTS + q] = m[q];
        ticket[o] = 0;
    }
}

// One row per atom: rho[2][N] (LDA: row 0 = total density, row 1 = 0), V[2][N] (LDA: row 1 = 0), V_H = U / r (node 0: 0, the value V
// holds there), and the electron count / <r^2> of the total density
__global__ void __launch_bounds__(kRT) radial_fields_kernel(GridDev g, ScfBuffers b, double* __restrict__ rho_out, double* __restrict__ v_out,
                                                            double* __restrict__ vh_out, double* __restrict__ atom_moments,
                                                            double* __restrict__ part, int* __restrict__ ticket)
{
    __shared__ double smem[2 * 32];
    const int a = blockIdx.x, N = g.N;
    const int ns = b.atoms[a].n_spin;
    const int t0 = b.tab_of[2 * a], t1 = ns == 2 ? b.tab_of[2 * a + 1] : -1;
    const double* U = b.U + (size_t)a * b.ldU;
    const double* rt = b.rhot + (size_t)a * N;
    double* ro = rho_out + (size_t)a * 2 * N;
    double* vo = v_out + (size_t)a * 2 * N;
    const int per = (N + (int)gridDim.y - 1) / (int)gridDim.y;
    const int i0 = blockIdx.y * per, i1 = min(i0 + per, N);
    double m[2] = { 0., 0. };
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        ro[i] = b.rho[(size_t)t0 * N + i];
        ro[N + i] = t1 >= 0 ? b.rho[(size_t)t1 * N + i] : 0.;
        vo[i] = b.vpot[(size_t)t0 * N + i];
        vo[N + i] = t1 >= 0 ? b.vpot[(size_t)t1 * N + i] : 0.;
        const double r = g.r[i];
        vh_out[(size_t)a * N + i] = i > 0 ? U[i] / r : 0.;
        const double w = kFourPi * g.wjac[i] * r * r * rt[i];
        m[0] += w;
        m[1] = fma(w, r * r, m[1]);
    }
    if (radial_finish<2>(m, part + (size_t)a * gridDim.y * 2, ticket + a, smem) && threadIdx.x == 0) {
        atom_moments[2 * a] = m[0];
        atom_moments[2 * a + 1] = m[1];
        ticket[a] = 0;
    }
}

long long radial_part_doubles(int N, int n_rows) { return (long long)n_rows * radial_chunks(N) * 3; }

void launch_radial_orbitals(const GridDev& g, const double* src, const double* inv_norm, int from_scf, int n_rows, double* u_out, double* moments,
                            double* part, int* ticket, cudaStream_t st)
{
    radial_orbitals_kernel<<<dim3(n_rows, radial_chunks(g.N)), kRT, 0, st>>>(g, src, inv_norm, from_scf, u_out, moments, part, ticket);
}

void launch_radial_fields(const GridDev& g, const ScfBuffers& b, double* rho_out, double* v_out, double* vh_out, double* atom_moments,
                          double* part, int* ticket, cudaStream_t st)
{
    radial_fields_kernel<<<dim3(b.n_atoms, radial_chunks(g.N)), kRT, 0, st>>>(g, b, rho_out, v_out, vh_out, atom_moments, part, ticket);
}

}  // namespace dft
