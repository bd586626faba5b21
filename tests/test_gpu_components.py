"""GPU parity tests of the component entry points (through the C ABI) against the CPU oracle on the same inputs."""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu


def _potential(kind, Z, r):
    V = np.zeros_like(r)
    if kind == "coulomb":
        V[1:] = -Z / r[1:]
    else:   # screened, with a bump: not monotone, exercises the turning-point logic
        V[1:] = -Z / r[1:] * (0.35 + 0.65 * np.exp(-1.3 * r[1:])) + 1.5 * np.exp(-0.4 * r[1:])
    return V


@pytest.mark.parametrize("kind,L,delta,rmax,Z", [("coulomb", 12, 0.001, 15.0, 18), ("screened", 13, 0.0008, 30.0, 64),
                                                 ("coulomb", 10, 0.004, 15.0, 92), ("screened", 20, 1.25e-5, 50.0, 36)])
def test_numerov_lanes_match_oracle(ctx, kind, L, delta, rmax, Z):
    """(sign y0, node count) of SolutionInZero / CountNodes: bit-exact except where |y0| is at its rounding floor."""
    N, rp, r = O.grid(L, delta, rmax)
    V = _potential(kind, Z, r)
    rng = np.random.default_rng(L)
    n_l = 384
    ls = rng.integers(0, 4, n_l).astype(np.int32)
    Es = np.concatenate([-10 ** rng.uniform(-2, np.log10(Z * Z + 1.0), n_l - 48), rng.uniform(0, 50, 48)])
    lim = rng.integers(0, 6, n_l).astype(np.int32)
    y0, cnt_o = O.numerov_lanes(V, delta, rmax, ls, Es, lim)
    # reference-shaped sweep: CountNodes with its early exits
    sign, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, ls, Es, lim, impl=1)
    assert np.array_equal(cnt, cnt_o)
    assert np.array_equal(sign, (y0 > 0).astype(np.int32))
    # |y0| to ~1e-6 relative (1e15 guard needs a factor 2); at 1048577 nodes the rounding of the longer sweep: 4.4e-6 measured on a B200
    atol = 1e-6 if L <= 17 else 1e-5
    np.testing.assert_allclose(lg, np.log2(np.abs(y0)), atol=atol)
    # production tile-staged sweep: same y0, and the full Sturm count (all sign changes, no early exit)
    sign, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, ls, Es, lim, impl=0)
    assert np.array_equal(sign, (y0 > 0).astype(np.int32))
    np.testing.assert_allclose(lg, np.log2(np.abs(y0)), atol=atol)
    assert np.array_equal(cnt, O.numerov_count_all(V, delta, rmax, ls, Es))
    # the same through the parallel-in-r sweep (cluster per 32 lanes, 8 / 32 radial segments)
    try:
        for segs in (8, 32):
            ctx.set_option("r_segments", segs)
            sign, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, ls, Es, lim, impl=2)
            assert np.array_equal(sign, (y0 > 0).astype(np.int32))
            np.testing.assert_allclose(lg, np.log2(np.abs(y0)), atol=atol)
            assert np.array_equal(cnt, O.numerov_count_all(V, delta, rmax, ls, Es))
    finally:
        ctx.set_option("r_segments", -1)
    # the production sweep (numerov_rows.cu): lanes across the radial grid, 4 / 8 / 16 trial energies per round on 128 / 64 / 32 segments
    for impl in (4, 5, 6):
        sign, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, ls, Es, lim, impl=impl)
        assert np.array_equal(sign, (y0 > 0).astype(np.int32)), impl
        np.testing.assert_allclose(lg, np.log2(np.abs(y0)), atol=atol)
        assert np.array_equal(cnt, O.numerov_count_all(V, delta, rmax, ls, Es)), impl


def test_numerov_known_answer_hydrogenic(ctx):
    """V = -Z/r: y0(E) changes sign at E_n = -Z^2/2n^2; for l = 0 the node count steps from n-1 to n there (SURVEY C5b)."""
    L, delta, rmax, Z = 14, 0.0005, 25.0, 18
    N, rp, r = O.grid(L, delta, rmax)
    V = _potential("coulomb", Z, r)
    for n, l in [(1, 0), (2, 0), (2, 1), (3, 0), (3, 2), (4, 3)]:
        En = -Z * Z / (2.0 * n * n)
        E = np.array([En - 1e-3, En + 1e-3])
        for impl in (0, 1):
            sign, lg, cnt = ctx.numerov_lanes(V, L, delta, rmax, [l, l], E, [50, 50], impl=impl)
            assert sign[0] != sign[1]
            if l == 0 or impl == 0:
                off = 1 if (l == 3 and impl == 0) else 0
                assert (cnt[0], cnt[1]) == (n - l - 1 + off, n - l + off)


@pytest.mark.parametrize("kind,L,delta,rmax,Z", [("coulomb", 12, 0.001, 15.0, 18), ("screened", 13, 0.0008, 30.0, 64)])
def test_level_search_matches_oracle(ctx, kind, L, delta, rmax, Z):
    """Eigenvalues of the concurrent K-section search vs the reference's chained bisection: <= 1e-9 Ha (bar: 1e-6)."""
    N, rp, r = O.grid(L, delta, rmax)
    V = _potential(kind, Z, r)
    ns = [1, 2, 2, 3, 3, 3, 4, 4, 4, 4]
    ls = [0, 0, 1, 0, 1, 2, 0, 1, 2, 3]
    if kind == "screened":
        ns, ls = ns[:6], ls[:6]
    E_o, ok_o = O.level_search(V, delta, rmax, Z, ns, ls, chained=True)
    # search_mode 0: Sturm-count search with interpolated ladders (production) in its two shapes - serial in r (one warp
    # per orbital, r_segments <= 1) and parallel in r (one cluster per orbital, 8 / 32 radial segments);
    # search_mode 1: reference-shaped three-stage search
    # search_kernel 0 (production): lanes across the radial grid, 4 trial energies per thread (numerov_rows.cu); 1: lanes across 32 energies
    for kern, mode, segs in ((0, 0, -1), (1, 0, 0), (1, 0, 8), (1, 0, 32), (0, 1, 0)):
        ctx.set_option("search_kernel", kern)
        ctx.set_option("search_mode", mode)
        ctx.set_option("r_segments", segs)
        E_g, ok_g = ctx.level_search(V, L, delta, rmax, Z, ns, ls)
        ctx.set_option("search_kernel", 0)
        ctx.set_option("search_mode", 0)
        ctx.set_option("r_segments", -1)
        np.testing.assert_allclose(E_g, E_o, rtol=0, atol=5e-9)
        assert ok_g.tolist() == ok_o.tolist()
    if kind == "coulomb":
        np.testing.assert_allclose(E_g, [-Z * Z / (2.0 * n * n) for n in ns], atol=5e-5)


@pytest.mark.parametrize("L,delta,rmax,Z", [(12, 0.001, 15.0, 18), (16, 0.0002, 50.0, 30), (17, 0.0001, 50.0, 86), (18, 5e-5, 50.0, 54),
                                         (20, 1.25e-5, 50.0, 92)])
def test_orbital_matches_oracle(ctx, L, delta, rmax, Z):
    """Two-sided matched + normalised solution (Numerov.h:403-504, DFTAtom.cpp:36-56).  16, 17 levels: the grid does not fit
    in shared memory and the production kernel works through it window by window (match_win_kernel)."""
    N, rp, r = O.grid(L, delta, rmax)
    V = _potential("coulomb", Z, r)
    for n, l in [(1, 0), (2, 1), (3, 0), (3, 2), (4, 3)]:
        E = O.level_search(V, delta, rmax, Z, [n], [l], chained=False)[0][0] if l < 3 else -Z * Z / 32.0 - 1e-7
        u_o, mp_o = O.orbital(V, delta, rmax, l, E)
        # 0: CTA-wide segmented transfer-matrix solve out of shared memory (production), 2: the same by one warp,
        # 1: serial kernel in the reference's arithmetic
        for mode in (0, 2, 1):
            ctx.set_option("match_mode", mode)
            u_g, mp_g = ctx.numerov_orbital(V, L, delta, rmax, l, E)
            ctx.set_option("match_mode", 0)
            assert abs(mp_g - mp_o) <= (0 if mode == 1 else 1)      # the match point is an argmax: rounding may move it by one node
            # rounding accumulates with the number of nodes: 2e-10 observed at 131073 nodes (relative 1e-10); measured on a B200:
            # 4.8e-10 at 262145 nodes, 3.0e-9 at 1048577
            np.testing.assert_allclose(u_g, u_o, rtol=0, atol=1e-10 if L <= 14 else 1e-9 if L <= 18 else 1e-8)


@pytest.mark.parametrize("L,delta,rmax,stream", [(10, 0.004, 15.0, 0), (14, 0.0005, 25.0, 0), (16, 0.0002, 50.0, 0), (14, 0.0005, 25.0, 1),
                                                 (15, 0.0004, 50.0, 1), (16, 0.0002, 50.0, 1), (17, 0.0001, 50.0, 1), (18, 5e-5, 50.0, 0),
                                                 (18, 5e-5, 50.0, 1), (20, 1.25e-5, 50.0, 0), (20, 1.25e-5, 50.0, 1)])
def test_poisson_matches_oracle_and_analytic(ctx, L, delta, rmax, stream):
    """U(r) of FMG + V-cycles vs the reference algorithm (oracle, 100 V-cycles) and vs the analytic Hartree potential.
    stream: the solver for many densities on grids beyond the chip (poisson_stream.cu) instead of one CTA / team per density."""
    N, rp, r = O.grid(L, delta, rmax)
    Zs = [1, 18, 86]
    a = [0.8, 1.7, 3.1]
    rho = np.stack([Z * k ** 3 / np.pi * np.exp(-2 * k * r) for Z, k in zip(Zs, a)])
    ctx.set_option("stream_poisson", stream)
    ctx.set_option("stream_min_dens", 1)
    ctx.set_option("stream_min_levels", 14)
    try:
        U, used = ctx.poisson_solve(L, delta, rmax, Zs, rho)
    finally:
        ctx.set_option("stream_poisson", 1)
        ctx.set_option("stream_min_dens", 4)
        ctx.set_option("stream_min_levels", 15)
    assert (used <= 20).all() and (used >= 3).all()
    for j, (Z, k) in enumerate(zip(Zs, a)):
        U_o, errs = O.poisson(L, delta, rmax, Z, rho[j], max_vcycles=100 if L <= 14 else 12)
        U_x = Z * (1 - np.exp(-2 * k * r) * (1 + k * r))
        # both are the same discrete solution up to their FP64 rounding floors (SURVEY fact 3: 7e-10 at L=14), which grow like
        # eps N^1.5: above 17 levels the bars of 17 levels scaled so.  Measured on a B200, per unit of Z: 4.8e-9 at 18 levels, 4.7e-8 at 20
        # (bars 2.3e-8, 1.8e-7); the gap to the analytic potential 2.1e-9 at 18, 4.1e-8 at 20 (bars 2.8e-8, 2.3e-7)
        grow = max(1.0, (N / 131073.0) ** 1.5)
        assert np.max(np.abs(U[j] - U_o)) < 2e-9 * max(1, Z) * (4 if L > 14 else 1) * grow
        assert abs(np.max(np.abs(U[j] - U_x)) - np.max(np.abs(U_o - U_x))) < 1e-8 * Z * grow
        assert U[j][0] == 0.0 and U[j][-1] == Z


def test_poisson_vcycle_shape(ctx):
    """One reference-shaped V-cycle (3+3 lexicographic GS sweeps per level, injection, linear prolongation) from the same
    state gives the same iterate as the oracle: the parallel scan evaluates the same sweep."""
    L, delta = 12, 0.001
    N, rp, r = O.grid(L, delta, 15.0)
    rng = np.random.default_rng(3)
    src = np.zeros((2, N)); src[:, 1:-1] = rng.standard_normal((2, N - 2)) * 1e-3
    phi = np.zeros((2, N)); phi[:, -1] = [3.0, 40.0]
    g, err = ctx.poisson_vcycles(L, delta, phi, src, 1)
    for j in range(2):
        o, err_o = O.poisson_vcycles(L, delta, phi[j], src[j], 1)
        np.testing.assert_allclose(g[j], o, rtol=0, atol=1e-12 * np.max(np.abs(o)))
        assert abs(err[j] - err_o) <= 1e-9 * err_o + 1e-15


@pytest.mark.parametrize("L,delta,variant,mid", [(15, 0.0004, 0, 11), (15, 0.0004, 1, 12), (15, 0.0004, 2, 14), (16, 0.0002, 0, 11), (17, 0.0001, 0, 14)])
def test_poisson_stream_vcycles_match_oracle(ctx, L, delta, variant, mid):
    """Stream mode (config C5a's kernel: slab windows with halos over the levels above 16384 nodes, one launch per level visit
    of all densities, poisson_mid_kernel below): 1 and 3 V-cycles, with and without the fused 6-sweep top visit, give the
    oracle's iterate (PoissonSolver.h:155-159) from the same state."""
    import torch
    N = (1 << L) + 1
    ld = N + 3
    nd = 4
    rng = np.random.default_rng(L)
    r = np.arange(N) / (N - 1)
    src = np.zeros((nd, N)); phi = np.zeros((nd, N))
    src[0, 1:-1] = rng.standard_normal(N - 2) * 1e-3                       # rough: every level's restriction matters
    src[1, 1:-1] = 1e-6 * np.exp(-30 * r[1:-1]) * (1 + 0.1 * rng.standard_normal(N - 2))
    src[2, 1:-1] = 1e-7 * np.sin(40 * r[1:-1])
    src[3, 1:-1] = rng.standard_normal(N - 2) * 1e-4
    phi[:, -1] = [3.0, 40.0, 86.0, 1.0]
    phi[1, 1:-1] = 40.0 * r[1:-1] ** 2 + 1e-3 * rng.standard_normal(N - 2)  # large smooth starting iterate
    phi[3, 1:-1] = 1e-3 * rng.standard_normal(N - 2)                        # rough starting iterate
    ctx.set_option("stream_variant", variant)
    ctx.set_option("stream_mid_levels", mid)        # levels of up to 2^mid nodes: one CTA per density; above: slab windows
    sb = ctx.poisson_scratch_bytes(L, nd)
    scratch = torch.empty(sb // 8, dtype=torch.float64, device="cuda")
    d_src = torch.zeros((nd, ld), dtype=torch.float64, device="cuda")
    d_src[:, :N] = torch.from_numpy(src).cuda()
    # The residual 4 (S + Phi_{2i-1} - 2 Phi_{2i} + Phi_{2i+1}) cancels to ~1e-8 of |Phi| on a smooth iterate and the coarse-grid
    # correction applies ~A^-1 to it: two evaluations of the same cycle that differ in the last bit of Phi (scan order, FMA
    # contraction, the dense coarse operator) differ by ~eps N^1.5 |Phi| afterwards (SURVEY fact 3: the reference's own answer
    # is only accurate to 7e-10 at L = 14 .. 5.6e-8 at L = 17).  Densities whose interior starts at ~0 have no such cancellation
    # in the first cycle and must agree to 1e-11.
    loose = 8 * 2.2e-16 * float(N) ** 1.5
    try:
        for n_cycles, fuse in ((1, False), (3, True), (3, False)):
            d_phi = torch.zeros((nd, ld), dtype=torch.float64, device="cuda")
            d_phi[:, :N] = torch.from_numpy(phi).cuda()
            torch.cuda.synchronize()
            ms, nl = ctx.poisson_vcycles_dev(L, delta, nd, d_phi.data_ptr(), d_src.data_ptr(), ld, scratch.data_ptr(), sb, n_cycles, fuse)
            K = L - mid
            assert nl == n_cycles * (2 * K + 1) - (n_cycles - 1 if fuse else 0)
            g = d_phi[:, :N].cpu().numpy()
            for j in range(nd):
                o, _ = O.poisson_vcycles(L, delta, phi[j], src[j], n_cycles)
                scale = np.max(np.abs(o))
                tol = (1e-11 if (n_cycles == 1 and j != 1) else loose) * scale
                assert np.max(np.abs(g[j] - o)) <= tol, (n_cycles, fuse, j, np.max(np.abs(g[j] - o)), tol)
                assert g[j][0] == phi[j][0] and g[j][-1] == phi[j][-1]
    finally:
        ctx.set_option("stream_variant", 0)
        ctx.set_option("stream_mid_levels", 11)


def test_vwn_matches_oracle(ctx):
    rng = np.random.default_rng(0)
    rho = np.concatenate([10.0 ** rng.uniform(-20, 5, 4000), [0.0, 1e-19, 1e-18, 0.999e-18]])
    v, e = ctx.vwn(rho)
    v_o, e_o = O.vwn_lda(rho)
    # device libm (log, atan, pow) differs from glibc by an ulp or two and B.5 cancels between its terms
    np.testing.assert_allclose(v, v_o, rtol=2e-11, atol=1e-300)
    np.testing.assert_allclose(e, e_o, rtol=2e-11, atol=1e-300)
    rb = rho * rng.uniform(0, 1, len(rho))
    rb[:10] = 0.0                        # fully polarised: rs_beta = inf (H atom)
    for x, y in zip(ctx.vwn(rho, rb), O.vwn_lsda(rho, rb)):
        np.testing.assert_allclose(x, y, rtol=5e-10, atol=1e-300)


def test_simpson38_matches_oracle(ctx):
    rng = np.random.default_rng(1)
    for n in (5, 17, 1025, 16385):
        v = rng.standard_normal((3, n))
        out = ctx.simpson38(0.7, v)
        ref = np.array([O.simpson38(0.7, row) for row in v])
        np.testing.assert_allclose(out, ref, rtol=0, atol=1e-12 * np.sqrt(n))


def test_quadrature_family_matches_oracle(ctx):
    """dftatom_integrate: every rule of Integral.h as a block reduction against the oracle (summation order differs: 1e-13)."""
    rng = np.random.default_rng(2)
    for n in (5, 17, 129, 1025, 16385, 131073):
        v = rng.standard_normal((3, n))
        for rule in range(5):
            out = ctx.integrate(rule, 0.7, v)
            ref = np.array([O.integrate(rule, 0.7, row) for row in v])
            np.testing.assert_allclose(out, ref, rtol=0, atol=2e-13 * np.sqrt(n) * 32)
    x = np.linspace(0.0, 5.0, 16385)
    assert abs(ctx.integrate(4, x[1] - x[0], np.exp(-x))[0] - (1 - np.exp(-5.0))) < 1e-14
    with pytest.raises(Exception):
        ctx.integrate(3, 0.1, np.zeros(7))          # Boole needs 4k + 1 samples (Integral.h:78)


def test_chachiyo_matches_oracle(ctx):
    """dftatom_xc_lda: the Chachiyo functionals (ExcCor.h:27-95) against the oracle; functional 0 is the VWN path."""
    rng = np.random.default_rng(4)
    rho = np.concatenate([10.0 ** rng.uniform(-20, 5, 4000), [0.0, 1e-19, 1e-18, 0.999e-18]])
    for functional in (1, 2):
        v, e = ctx.xc_lda(functional, rho)
        v_o, e_o = O.xc_chachiyo(rho, functional - 1)
        np.testing.assert_allclose(v, v_o, rtol=2e-11, atol=1e-300)
        np.testing.assert_allclose(e, e_o, rtol=2e-11, atol=1e-300)
    v, e = ctx.xc_lda(0, rho)
    v_o, e_o = O.vwn_lda(rho)
    np.testing.assert_allclose(v, v_o, rtol=2e-11, atol=1e-300)


@pytest.mark.parametrize("L,rmax", [(12, 15.0), (14, 25.0), (15, 25.0)])
def test_poisson_uniform_grid_matches_oracle(ctx, L, rmax):
    """First kernel-level piece of the uniform-grid pair (SURVEY 8(f) rank 1): dftatom_poisson_solve with delta = 0 is
    SolvePoissonUniform (PoissonSolver.h:20-49: r_i = i h, no first-derivative term, source r h^2 4 pi rho) against the oracle
    and the analytic Hartree potential of an exponential density."""
    N = (1 << L) + 1
    r = np.arange(N) * (rmax / (N - 1))
    Zs = [1, 18, 86]
    a = [0.8, 1.7, 3.1]
    rho = np.stack([Z * k ** 3 / np.pi * np.exp(-2 * k * r) for Z, k in zip(Zs, a)])
    ctx.set_option("stream_min_dens", 1)
    try:
        U, used = ctx.poisson_solve(L, 0.0, rmax, Zs, rho)
    finally:
        ctx.set_option("stream_min_dens", 4)
    for j, (Z, k) in enumerate(zip(Zs, a)):
        U_o = O.poisson_uniform(L, rmax, Z, rho[j], max_vcycles=100 if L <= 14 else 12)
        U_x = Z * (1 - np.exp(-2 * k * r) * (1 + k * r))
        assert np.max(np.abs(U[j] - U_o)) < 2e-9 * max(1, Z) * (4 if L > 14 else 1)
        assert abs(np.max(np.abs(U[j] - U_x)) - np.max(np.abs(U_o - U_x))) < 1e-8 * Z
        assert U[j][0] == 0.0 and U[j][-1] == Z



@pytest.mark.parametrize("L,delta,rmax", [(8, 0.02, 10.0), (10, 0.004, 15.0), (14, 0.0005, 25.0), (16, 0.0002, 50.0), (17, 0.0001, 50.0),
                                          (18, 5e-5, 50.0), (20, 1.25e-5, 50.0), (12, 0.0, 15.0), (14, 0.0, 25.0)])
def test_poisson_exact_mode_is_bit_identical(ctx, L, delta, rmax):
    """set_option("poisson_exact", 1): the reference's FullCycle (Initialize, FMG ramp with its 1e-3 early exits, 100 V-cycles) in the
    reference's own floating-point operation order (PoissonSolver.cpp:40-157, .h:51-124), chunk-parallel with a 128-node warm-up halo:
    U(r) must equal the CPU solver's BIT FOR BIT - against the C restatement and, where oracle/_ref was built, against the unmodified
    reference's own PoissonSolver class.  delta = 0: SolvePoissonUniform (.h:20-49)."""
    N = (1 << L) + 1
    if delta > 0:
        _, rp, r = O.grid(L, delta, rmax)
    else:
        r = np.arange(N) * (rmax / (N - 1))
    Zs = [1, 18, 86]
    rng = np.random.default_rng(L)
    # shell-like densities with rough (non-smooth) multiplicative noise: the bits must agree whatever the input
    rho = np.stack([Z * k ** 3 / np.pi * np.exp(-2 * k * r) * (1 + 1e-3 * rng.standard_normal(N)) for Z, k in zip(Zs, [0.8, 1.7, 3.1])])
    ctx.set_option("poisson_exact", 1)
    try:
        U, used = ctx.poisson_solve(L, delta, rmax, Zs, rho)
    finally:
        ctx.set_option("poisson_exact", 0)
    ref = O.ref_components()
    for j, Z in enumerate(Zs):
        if delta > 0:
            U_o, errs = O.poisson(L, delta, rmax, Z, rho[j], max_vcycles=100)
            assert used[j] == len(errs)
        else:
            U_o = O.poisson_uniform(L, rmax, Z, rho[j], max_vcycles=100)
        assert np.array_equal(U[j], U_o), (L, Z, np.max(np.abs(U[j] - U_o)))
        if ref is not None and delta > 0:
            U_r = np.zeros(N)
            ref.ref_poisson_nonuniform(L, delta, int(Z), rmax, O.d(np.ascontiguousarray(rho[j])), O.d(U_r))
            assert np.array_equal(U[j], U_r)


@pytest.mark.parametrize("kind,L,delta,rmax,Z", [("coulomb", 12, 0.001, 15.0, 18), ("screened", 13, 0.0008, 30.0, 64)])
def test_outward_node_count_matches_oracle(ctx, kind, L, delta, rmax, Z):
    """SURVEY 8(f) rank 4: SolveSchrodingerCountNodesFromNucleus (Numerov.h:204-270; public in the reference, no caller) as lanes
    (impl = 3): the count of the outward sweep with its three early exits, bit-exact against the oracle's restatement (itself pinned on
    the reference's own class in tests/test_oracle.py) on random (l, E, limit) lanes incl. positive energies."""
    N, rp, r = O.grid(L, delta, rmax)
    V = _potential(kind, Z, r)
    rng = np.random.default_rng(7 * L)
    n_l = 256
    ls = rng.integers(0, 4, n_l).astype(np.int32)
    Es = np.concatenate([-10 ** rng.uniform(-2, np.log10(Z * Z + 1.0), n_l - 32), rng.uniform(0, 50, 32)])
    lim = rng.integers(0, 7, n_l).astype(np.int32)
    _, _, cnt = ctx.numerov_lanes(V, L, delta, rmax, ls, Es, lim, impl=3)
    assert np.array_equal(cnt, O.numerov_count_from_nucleus(V, delta, rmax, ls, Es, lim))
    # known answer: in a Coulomb well the outward count up to the outer turning point of E just above E_n (l = 0) is n - 1... n
    if kind == "coulomb":
        E3 = -Z * Z / 18.0
        _, _, c3 = ctx.numerov_lanes(V, L, delta, rmax, np.zeros(2, np.int32), np.array([E3 * 1.02, E3 * 0.98]), np.full(2, 10, np.int32), impl=3)
        assert list(c3) == [2, 2] or list(c3) == [2, 3]
