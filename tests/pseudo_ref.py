"""numpy reference of dftatom_tm_pseudize (definition: include/dftatom_b200.h): Troullier-Martins pseudization of one channel, and the
unscreening of the channels that share a potential row.

The all-electron data at r_c come from the outward sweep of logderiv_ref.py at E = eps.  The coefficients are solved in the scaled
variable t = r / r_c (d_2k = c_2k r_c^2k, x = d_2); the norm F(x) = ln S(x) - ln q is searched on the ladder x = 0, -1/2, +1/2, ... and
refined by 8-point multisection, keeping the sub-interval nearest x = 0, as the kernel does.  V_H comes from scipy's banded solve of the
multigrid's level-0 system -(1 + delta/2) U_(i-1) + 2 U_i - (1 - delta/2) U_(i+1) = 4 pi r_i K_i rho_i, U_0 = 0, U_(N-1) = Q."""
import numpy as np
from scipy.linalg import solve_banded

import logderiv_ref as LR

LADDER = 128
REL_TOL = 1e-13
MAX_REFINE = 40
POINTS = 8                     # candidates per multisection round
_M = np.array([[6., 8., 10., 12.], [30., 56., 90., 132.], [120., 336., 720., 1320.], [360., 1680., 5040., 11880.]])


def ae_data(V, levels, delta, max_r, l, eps, u_row, r_c):
    """i_c, r_c used, D and u_n(r_c) of the sweep at eps, a, s, q, the derivative targets p, p', .., p'''' at r_c and the sweep flag."""
    N, r, _, _ = LR.grid(levels, delta, max_r)
    n = LR.nearest_node(r, r_c)
    Dv, un, _, nodes, rc = LR.log_derivative(V, levels, delta, max_r, l, r_c, [eps])
    a = abs(u_row[n])
    s = -1.0 if u_row[n] < 0 else 1.0
    bad = nodes[0] < 0
    q = a * a / (un[0] * un[0])
    vi1 = ((V[n - 2] - 8 * V[n - 1]) + (8 * V[n + 1] - V[n + 2])) / 12
    vi2 = (((-V[n - 2] + 16 * V[n - 1]) - 30 * V[n]) + (16 * V[n + 1] - V[n + 2])) / 12
    if delta == 0.0:
        J = max_r / (N - 1)
    else:
        rp = max_r / (np.exp((N - 1) * delta) - 1.0)
        J = delta * (rc + rp)
    v1, v2 = vi1 / J, (vi2 - delta * vi1) / (J * J)
    L1 = l + 1.0
    p1 = Dv[0] - L1 / rc
    p2 = 2 * (V[n] - eps) - 2 * L1 * p1 / rc - p1 * p1
    p3 = 2 * v1 + 2 * L1 * p1 / rc ** 2 - 2 * L1 * p2 / rc - 2 * p1 * p2
    p4 = 2 * v2 - 4 * L1 * p1 / rc ** 3 + 4 * L1 * p2 / rc ** 2 - 2 * L1 * p3 / rc - 2 * p2 * p2 - 2 * p1 * p3
    p0 = np.log(a / rc ** (l + 1))
    return dict(n=n, r_c=rc, D=Dv[0], u_n=un[0], a=a, s=s, q=q, bad=bad, p=(p0, p1, p2, p3, p4))


def coeff_vectors(ae, l):
    """(A, B, C): (d6, d8, d10, d12) = A + x B + x^2 C."""
    rc = ae["r_c"]
    _, p1, p2, p3, p4 = ae["p"]
    T = np.array([rc * p1, rc ** 2 * p2, rc ** 3 * p3, rc ** 4 * p4])
    X = np.linalg.solve(_M, np.column_stack([T, [2., 2., 0., 0.], [4., 12., 24., 24.]]))
    return X[:, 0], -X[:, 1], X[:, 2] / (2 * l + 5)


def scaled_coeffs(ae, l, x, vecs=None):
    """d0 .. d12 at x."""
    A, B, C = coeff_vectors(ae, l) if vecs is None else vecs
    d = np.zeros(7)
    d[1] = x
    d[2] = -(x * x) / (2 * l + 5)
    d[3:] = A + x * (B + x * C)
    d[0] = ae["p"][0] - (d[1] + d[2] + d[3] + d[4] + d[5] + d[6])
    return d


def _p(d, t2):
    return np.polynomial.polynomial.polyval(t2, d)


def norm_F(ae, l, x, r, jac, vecs):
    n = ae["n"]
    d = scaled_coeffs(ae, l, x, vecs)
    rr = r[:n + 1]
    with np.errstate(over="ignore", invalid="ignore"):
        u = rr ** (l + 1) * np.exp(_p(d, (rr / ae["r_c"]) ** 2))
        return np.log(np.sum(LR.simpson_weights(n) * u * u * jac[:n + 1])) - np.log(ae["q"])


def _changes(fa, fb):
    return (fa <= 0 and fb >= 0) or (fa >= 0 and fb <= 0)


def find_root(ae, l, r, jac):
    """(x, status): x = c2 r_c^2 of the definition's root and status 0; (None, 1) without a sign change on the ladder; (None, 3) when the
    multisection stops short of 1e-13 (no sub-interval changes sign, or MAX_REFINE rounds)."""
    vecs = coeff_vectors(ae, l)
    F = {}

    def f(x):
        if x not in F:
            F[x] = norm_F(ae, l, x, r, jac, vecs)
        return F[x]
    bracket = None
    for k in range(1, LADDER + 1):
        for xa, xb in ((-0.5 * k, -0.5 * (k - 1)), (0.5 * (k - 1), 0.5 * k)):
            if _changes(f(xa), f(xb)):
                bracket = (xa, xb)
                break
        if bracket:
            break
    if bracket is None:
        return None, 1
    lo, hi = bracket
    flo, fhi = f(lo), f(hi)
    for rnd in range(MAX_REFINE):
        xs = [lo] + [lo + (hi - lo) * ((j + 1) * (1.0 / (POINTS + 1))) for j in range(POINTS)] + [hi]
        fs = [flo] + [norm_F(ae, l, x, r, jac, vecs) for x in xs[1:-1]] + [fhi]
        idx = range(POINTS, -1, -1) if hi <= 0 else range(POINTS + 1)
        old = (lo, hi)
        for k in idx:
            if _changes(fs[k], fs[k + 1]):
                lo, hi, flo, fhi = xs[k], xs[k + 1], fs[k], fs[k + 1]
                break
        if hi - lo <= REL_TOL * max(abs(lo), abs(hi)):
            return 0.5 * (lo + hi), 0
        if (lo, hi) == old:
            break
    return None, 3


def tm_channel(V, u_row, levels, delta, max_r, l, eps, r_c):
    """One channel: dict(c [7] natural units, d [7] scaled, x, r_c, q, status, u_ps [N], v_scr [N], n)."""
    N, r, _, jac = LR.grid(levels, delta, max_r)
    V = np.asarray(V, np.float64)
    u_row = np.asarray(u_row, np.float64)
    ae = ae_data(V, levels, delta, max_r, l, eps, u_row, r_c)
    n, rc = ae["n"], ae["r_c"]
    x, status = (None, 2) if ae["bad"] else find_root(ae, l, r, jac)
    d = np.full(7, np.nan) if status else scaled_coeffs(ae, l, x)
    c = d / rc ** (2 * np.arange(7))
    u_ps = np.zeros(N)
    v_scr = np.zeros(N)
    ri = r[1:n + 1]
    t2 = (ri / rc) ** 2
    u_ps[1:n + 1] = ri ** (l + 1) * np.exp(_p(d, t2))
    k = np.arange(1, 7)
    q = _p(2 * k * d[1:], t2) / rc ** 2                         # p'/r
    p2 = _p(2 * k * (2 * k - 1) * d[1:], t2) / rc ** 2          # p''
    v_scr[1:n + 1] = eps + 0.5 * ((p2 + ri * ri * q * q) + 2 * (l + 1) * q)
    u_ps[n + 1:] = ae["s"] * u_row[n + 1:]
    v_scr[n + 1:] = V[n + 1:]
    return dict(c=c, d=d, x=x, r_c=rc, q=np.nan if ae["bad"] else ae["q"], status=status, u_ps=u_ps, v_scr=v_scr, n=n, ae=ae)


def hartree_U(levels, delta, max_r, rho, Q):
    """U = r V_H of the level-0 system of the multigrid Poisson solve, U_0 = 0, U_(N-1) = Q."""
    N, r, K, _ = LR.grid(levels, delta, max_r)
    S = r * (4 * np.pi * K) * rho
    m = N - 2
    ab = np.zeros((3, m))
    ab[0, 1:] = -(1 - 0.5 * delta)
    ab[1, :] = 2.0
    ab[2, :-1] = -(1 + 0.5 * delta)
    b = S[1:N - 1].copy()
    b[-1] += (1 - 0.5 * delta) * Q
    U = np.zeros(N)
    U[1:N - 1] = solve_banded((1, 1), ab, b)
    U[N - 1] = Q
    return U


def vwn_lda(rho):
    """V_xc of the spin-unpolarised VWN LDA of the SCF (0 below 1e-18)."""
    rho = np.asarray(rho, np.float64)
    out = np.zeros_like(rho)
    ok = rho >= 1e-18
    rs = np.cbrt(3.0 / (4 * np.pi * rho[ok]))
    A, y0, b, c = 0.0310907, -0.10498, 3.72744, 12.93532
    y = np.sqrt(rs)
    Y = y * (y + b) + c
    Y0 = y0 * y0 + b * y0 + c
    dy = y - y0
    Qq = np.sqrt(4 * c - b * b)
    at = np.arctan(Qq / (2 * y + b))
    eps = A * (np.log(y * y / Y) + 2 * b / Qq * at - b * y0 / Y0 * (np.log(dy * dy / Y) + 2 * (b + 2 * y0) / Qq * at))
    deps = A * (c * dy - b * y0 * y) / (dy * Y)
    x1 = 0.6108870577108572
    out[ok] = -x1 / rs + eps - deps / 3
    return out


def unscreen(levels, delta, max_r, channels):
    """channels: list of (tm_channel result, l, occ) of one potential row -> (rho_v [N], V_H [N], V_xc [N], [V_ion [N] per channel])."""
    N, r, _, _ = LR.grid(levels, delta, max_r)
    inv4pr2 = np.zeros(N)
    inv4pr2[1:] = 1.0 / (4 * np.pi * r[1:] ** 2)
    if any(ch["status"] for ch, _, _ in channels):
        nanrow = np.full(N, np.nan)
        nanrow[0] = 0.0
        return nanrow, None, None, [nanrow.copy() for _ in channels]
    acc = np.zeros(N)
    for ch, _, occ in channels:
        acc = acc + occ * ch["u_ps"] ** 2
    rho = acc * inv4pr2
    Q = sum(occ for _, _, occ in channels)
    vh = np.zeros(N)
    if Q > 0:
        U = hartree_U(levels, delta, max_r, rho, Q)
        vh[1:] = U[1:] / r[1:]
    vxc = vwn_lda(rho)
    vion = []
    for ch, _, _ in channels:
        v = ch["v_scr"] - vh - vxc
        v[0] = 0.0
        vion.append(v)
    return rho, vh, vxc, vion
