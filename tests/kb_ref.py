"""numpy / scipy reference of the Kleinman-Bylander calls dftatom_kb_form and dftatom_kb_log_derivatives (definitions:
include/dftatom_b200.h), with the discretisation, rescaling and quadrature of the engine, plus an independent ghost check: the
eigenvalues of the KB Hamiltonian as a dense matrix (second-order differences in the index variable, box u(max_r) = 0)."""
import numpy as np
from scipy.linalg import eigh

import logderiv_ref as LR

_BIG = 2.0 ** 128
_DOWN = 2.0 ** -256


def tables(levels, delta, max_r):
    """(N, r, K, jac, sqex, wjac): LR.grid plus e^(delta i / 2) and the radial export's Simpson38 weights times dr/di."""
    N, r, K, jac = LR.grid(levels, delta, max_r)
    i = np.arange(N)
    sqex = np.ones(N) if delta == 0.0 else np.exp(i * delta * 0.5)
    w = np.where((i == 0) | (i == N - 1), 1.0, np.where(i % 3 == 0, 2.0, 3.0))
    return N, r, K, jac, sqex, 0.375 * w * jac


def kb_form(V, u, levels, delta, max_r, row, loc, l, eps):
    """E_KB, cos, beta, i_s, r_s, status of one channel (dftatom_kb_form without the local eigenvalues)."""
    N, r, K, jac, sqex, wjac = tables(levels, delta, max_r)
    ur = np.asarray(u[row], np.float64)
    out = dict(i_s=0, r_s=0.0, beta=np.zeros(N))
    if row == loc:
        return dict(out, E_KB=0.0, cos=1.0, status=1)
    dv = np.zeros(N)
    dv[1:] = V[row][1:] - V[loc][1:]
    nz = np.nonzero(dv)[0]
    i_s = int(nz[-1]) if len(nz) else 0
    out.update(i_s=i_s, r_s=r[i_s])
    w = np.zeros(N)
    w[:i_s + 1] = LR.simpson_weights(i_s) * jac[:i_s + 1]
    a = np.sum(w * ur * ur * dv)
    b = np.sum(w * ur * ur * dv * dv)
    if a == 0.0 or i_s < 3:
        return dict(out, E_KB=np.nan, cos=np.nan, status=2)
    uu = np.sum(wjac * ur * ur)
    return dict(out, E_KB=b / a, cos=a / np.sqrt(uu * b), beta=dv * ur / np.sqrt(b), status=0)


def gss_ghost(E_KB, eps, eps_loc):
    """The Gonze-Stumpf-Scheffler verdict for a nodeless reference state: a ghost below eps."""
    return int(eps > eps_loc[1]) if E_KB > 0 else int(eps > eps_loc[0])


def _g(V, levels, delta, max_r, l):
    N, r, K, jac = LR.grid(levels, delta, max_r)
    rr = np.where(r > 0, r, 1.0)
    return (2.0 * K * V + np.where(r > 0, K * l * (l + 1) / rr ** 2, 0.0) + delta * delta / 4.0) / 12.0, K / 6.0


def outward(V, levels, delta, max_r, l, E, n):
    """y_0..y_n of the outward homogeneous sweep of dftatom_log_derivatives at one energy (no rescaling: for moderate n and E)."""
    N, r, K, jac = LR.grid(levels, delta, max_r)
    g0, gE = _g(np.asarray(V, np.float64), levels, delta, max_r, l)
    g = g0 - E * gE
    y = np.zeros(n + 1)
    y[1] = (max_r / (N - 1)) ** (l + 1) if delta == 0.0 else r[1] ** (l + 1) * np.exp(-0.5 * delta)
    wprev, w = 0.0, (1.0 - g[1]) * y[1]
    for i in range(2, n + 1):
        wn = 2.0 * w - wprev + 12.0 * g[i - 1] * y[i - 1]
        wprev, w = w, wn
        y[i] = wn / (1.0 - g[i])
    return y


def local_levels(V, levels, delta, max_r, l, k=2, tol=1e-13):
    """The k lowest eigenvalues of -1/2 u'' + [V + l(l+1)/2r^2] u, u(max_r) = 0, on the engine's grid: bisection on the Sturm count
    (sign changes of the outward Numerov solution over nodes 1..N-1)."""
    N, r, K, jac = LR.grid(levels, delta, max_r)
    g0, gE = _g(np.asarray(V, np.float64), levels, delta, max_r, l)
    y1 = (max_r / (N - 1)) ** (l + 1) if delta == 0.0 else r[1] ** (l + 1) * np.exp(-0.5 * delta)

    def count(E):
        g = g0 - E * gE
        y, wprev, w, c, pos = y1, 0.0, (1.0 - g[1]) * y1, 0, True
        for i in range(2, N):
            wn = 2.0 * w - wprev + 12.0 * g[i - 1] * y
            wprev, w = w, wn
            y = wn / (1.0 - g[i])
            if (pos and y < 0) or (not pos and y > 0):
                c += 1; pos = not pos
            if abs(y) > _BIG:
                y *= _DOWN; w *= _DOWN; wprev *= _DOWN
        return c

    lo0 = float(np.min(V[1:])) - 1.0
    out = []
    for want in range(k):
        lo, hi = lo0, 50.0
        while hi - lo > tol * max(1.0, abs(lo)):
            mid = 0.5 * (lo + hi)
            if count(mid) > want:
                hi = mid
            else:
                lo = mid
        out.append(0.5 * (lo + hi))
    return np.array(out)


def kb_log_derivative(V_loc, beta, levels, delta, max_r, l, E_KB, r_c, E, return_cond=False):
    """D, u, du, nodes ([n_energies]) and the radius used for one channel with projector beta (dftatom_kb_log_derivatives): the two
    chains of the definition to max(i_c, i_s) + 1 with their own power-of-two rescaling, combined as (sigma - E_KB h_p) u_h + E_KB h_h u_p;
    the node count from the combination at every node (kept per node here).  return_cond: also the condition number of the combination
    at r_c, ((|sigma| + |E_KB h_p|) |u_h| + |B u_p|) / |u|, by which it amplifies the rounding of the two sweeps and of A = sigma - E_KB h_p."""
    N, r, K, jac, sqex, _ = tables(levels, delta, max_r)
    n = LR.nearest_node(r, r_c)
    E = np.atleast_1d(np.asarray(E, np.float64))
    beta = np.asarray(beta, np.float64)
    nz = np.nonzero(beta)[0]
    ns = int(nz[-1]) if len(nz) else 0
    uniform = delta == 0.0
    src = 2.0 * K * beta if uniform else 2.0 * K * beta / sqex
    hw = np.zeros(N)
    hw[:ns + 1] = LR.simpson_weights(ns) * (jac * sqex * beta)[:ns + 1] if ns > 0 else 0.0
    wn_ = LR.simpson_weights(n) * 2.0 * K[:n + 1]
    g0, gE = _g(np.asarray(V_loc, np.float64), levels, delta, max_r, l)
    y1 = (max_r / (N - 1)) ** (l + 1) if uniform else r[1] ** (l + 1) * np.exp(-0.5 * delta)
    m = len(E)
    yh = np.full(m, y1); wh = (1.0 - (g0[1] - E * gE[1])) * y1; whp = np.zeros(m)
    yp = np.zeros(m); wp = np.zeros(m); wpp = np.zeros(m)
    sig = np.ones(m)
    hh = hw[1] * yh; hp = np.zeros(m)
    Shh = wn_[1] * yh * yh; Shp = np.zeros(m); Spp = np.zeros(m)
    bad = np.zeros(m, bool)
    YH = {1: yh.copy()}; YP = {1: yp.copy()}               # per node, at the scale of the node (scale exponents alongside)
    EH = {1: np.zeros(m, int)}; EP = {1: np.zeros(m, int)}
    eh = np.zeros(m, int); ep = np.zeros(m, int)
    g = g0[1] - E * gE[1]
    gs = {1: g}
    for i in range(2, max(n, ns) + 2):
        gi = g0[i] - E * gE[i]
        src3 = ((10.0 * src[i - 1] + src[i - 2]) + src[i]) * (1.0 / 12.0)
        wnh = 2.0 * wh - whp + 12.0 * g * yh
        wnp = sig * src3 + (2.0 * wp - wpp + 12.0 * g * yp)
        d = 1.0 - gi
        bad |= ~(d > 0)
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            rd = 1.0 / d
            whp, wh, wpp, wp = wh, wnh, wp, wnp
            yh, yp = wnh * rd, wnp * rd
        g = gi
        if i <= ns:
            hh = hh + hw[i] * yh; hp = hp + hw[i] * yp
        if i <= n:
            Shh = Shh + wn_[i] * yh * yh; Shp = Shp + wn_[i] * yh * yp; Spp = Spp + wn_[i] * yp * yp
        if (i & 7) == 1:
            bh = np.abs(yh) > _BIG
            yh = np.where(bh, yh * _DOWN, yh); wh = np.where(bh, wh * _DOWN, wh); whp = np.where(bh, whp * _DOWN, whp)
            hh = np.where(bh, hh * _DOWN, hh); Shh = np.where(bh, Shh * _DOWN * _DOWN, Shh); Shp = np.where(bh, Shp * _DOWN, Shp)
            eh = eh + bh
            bp = np.abs(yp) > _BIG
            yp = np.where(bp, yp * _DOWN, yp); wp = np.where(bp, wp * _DOWN, wp); wpp = np.where(bp, wpp * _DOWN, wpp)
            sig = np.where(bp, sig * _DOWN, sig); hp = np.where(bp, hp * _DOWN, hp)
            Spp = np.where(bp, Spp * _DOWN * _DOWN, Spp); Shp = np.where(bp, Shp * _DOWN, Shp)
            ep = ep + bp
        if i <= n + 1:
            YH[i], YP[i], EH[i], EP[i], gs[i] = yh.copy(), yp.copy(), eh.copy(), ep.copy(), g
    A = sig - E_KB * hp
    B = E_KB * hh

    def at(i, Y, Ei, efin):                                 # y at node i in the chain's final scale
        return np.ldexp(Y[i], -256 * (efin - Ei[i]))
    comb = {i: A * at(i, YH, EH, eh) + B * at(i, YP, EP, ep) for i in range(1, n + 2)}
    nodes = np.zeros(m, int)
    first = np.sign(A)
    cur = first.copy()
    for i in range(2, n + 1):
        # the sign of the combination in the scales of node i (one term may underflow in the final scales)
        dd = (eh - EH[i]) - (ep - EP[i])
        x, z = A * YH[i], B * YP[i]
        v = np.where(dd >= 0, x * np.ldexp(1.0, -256 * np.maximum(dd, 0)) + z, x + z * np.ldexp(1.0, -256 * np.maximum(-dd, 0)))
        s = np.sign(v)
        flip = (s != 0) & (cur != 0) & (s != cur)
        nodes += flip
        cur = np.where(s != 0, s, cur)
        first = np.where((first == 0) & (s != 0), s, first)
    dy = 0.5 * ((1.0 - 2.0 * gs[n + 1]) * comb[n + 1] - (1.0 - 2.0 * gs[n - 1]) * comb[n - 1]) - B * sig * (src[n + 1] - src[n - 1]) / 12.0
    s = A * A * Shh + 2.0 * A * B * Shp + B * B * Spp
    if uniform:
        h = max_r / (N - 1)
        uc, du, jac2 = comb[n], dy / h, 2.0 * h
    else:
        rp = max_r / (np.exp((N - 1) * delta) - 1.0)
        uc = comb[n] * sqex[n]
        du = (dy + 0.5 * delta * comb[n]) / (sqex[n] * rp * delta)
        jac2 = 2.0 * rp * delta
    with np.errstate(invalid="ignore", divide="ignore"):
        inv = np.where(first < 0, -1.0, 1.0) / np.sqrt(s / jac2)
        D, u, du = du / uc, uc * inv, du * inv
    nodes = np.where(bad, -1, nodes)
    D, u, du = (np.where(bad, np.nan, x) for x in (D, u, du))
    if return_cond:
        with np.errstate(invalid="ignore", divide="ignore"):
            cond = ((np.abs(sig) + np.abs(E_KB * hp)) * np.abs(at(n, YH, EH, eh)) + np.abs(B * at(n, YP, EP, ep))) / np.abs(comb[n])
        return D, u, du, nodes, r[n], cond
    return D, u, du, nodes, r[n]


def dense_kb_levels(V_loc, beta, levels, delta, max_r, l, E_KB, coarse_levels=11, k=6):
    """The k lowest eigenvalues of the KB Hamiltonian -1/2 u'' + [V_loc + l(l+1)/2r^2] u + E_KB beta <beta|u>, u(0) = u(max_r) = 0, as a
    dense matrix on every 2^(levels - coarse_levels)-th node of the grid (a grid of the same family with 2^coarse_levels + 1 nodes).
    In y = u / sqrt(dr/di): -1/2 y'' + [K V_eff + delta^2 / 8] y + E_KB b b^T y = E K y, b_i = (dr/di)^(3/2) beta_i, second-order
    differences in the index, <beta|u> as the plain sum over nodes."""
    s = 2 ** (levels - coarse_levels)
    N, r, K, jac = LR.grid(levels, delta, max_r)
    idx = np.arange(0, N, s)
    dl = delta * s
    rc, Kc, jc = r[idx], (jac[idx] * s) ** 2, jac[idx] * s
    inner = slice(1, len(idx) - 1)
    veff = np.asarray(V_loc, np.float64)[idx][inner] + l * (l + 1) / (2.0 * rc[inner] ** 2)
    n = len(idx) - 2
    H = np.diag(1.0 + Kc[inner] * veff + dl * dl / 8.0) - 0.5 * (np.eye(n, k=1) + np.eye(n, k=-1))
    b = jc[inner] ** 1.5 * np.asarray(beta, np.float64)[idx][inner]
    H += E_KB * np.outer(b, b)
    return eigh(H, np.diag(Kc[inner]), eigvals_only=True, subset_by_index=[0, k - 1])


def dense_ghost(V_loc, beta, levels, delta, max_r, l, E_KB, eps, margin, **kw):
    """1 if the dense KB Hamiltonian has an eigenvalue below eps - margin (a ghost below the reference level), else 0."""
    return int(dense_kb_levels(V_loc, beta, levels, delta, max_r, l, E_KB, **kw)[0] < eps - margin)
