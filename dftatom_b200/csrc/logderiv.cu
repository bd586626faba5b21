// Logarithmic derivatives D_l(E) = u'(r_c) / u(r_c) of the outward radial solution, batched over (channel, energy) lanes
// (dftatom_log_derivatives, include/dftatom_b200.h).  The pseudopotential diagnostic: D on an energy grid for every l, and the
// norm integral of u up to r_c for the identity dD/dE = -2 int_0^rc u^2 dr / u(r_c)^2.
//
// Every lane is one outward sweep from the nucleus over the SCF's own tables (logderiv_sweep.cuh).
//
// Shape: one warp = 32 energies of one channel, so every lane reads the same node's atab / b12 / c6 / k2 (warp-uniform loads);
// warps are dealt longest sweep first (the host orders `warp_item`).
#include "logderiv_sweep.cuh"

namespace dft {

__global__ void __launch_bounds__(128) logderiv_kernel(GridDev g, LogDerivArgs a)
{
    const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (warp >= a.n_warps) return;
    const int item = a.warp_item[warp];
    const int ch = item / a.energy_blocks;
    const int e = (item - ch * a.energy_blocks) * 32 + (threadIdx.x & 31);
    const double E = a.E[min(e, a.n_energies - 1)];      // tail lanes repeat the last energy and write nothing
    const dftatom_logderiv o = logderiv_sweep(g, a.atab + (size_t)a.pot[ch] * g.N, a.l[ch], a.ic[ch], E);
    if (e < a.n_energies) a.out[(size_t)ch * a.n_energies + e] = o;
}

void launch_logderiv(const GridDev& g, const LogDerivArgs& a, cudaStream_t st)
{
    logderiv_kernel<<<(a.n_warps + 3) / 4, 128, 0, st>>>(g, a);
}

}  // namespace dft
