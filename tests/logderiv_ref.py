"""numpy reference of the logarithmic derivatives of dftatom_log_derivatives (definition: include/dftatom_b200.h).

One outward Numerov sweep per energy, vectorised over the energies of one channel, in the operation order of the definition:
g_i = (2 K_i (V_i - E) + K_i l(l+1) / r_i^2 + delta^2 / 4) / 12, y_0 = 0, y_1 = r_1^(l+1) e^(-delta/2) (uniform grid: h^(l+1)),
w = (1 - g) y, w_(i+1) = 2 w_i - w_(i-1) + 12 g_i y_i, to node i_c + 1; Simpson 1/3 (3/8 on the last three intervals for odd i_c) for
int_0^rc u^2 dr; the fourth-order index derivative at i_c.  The sweep is rescaled by powers of two, so every lane stays finite."""
import numpy as np

_BIG = 2.0 ** 128
_DOWN = 2.0 ** -256


def grid(levels, delta, max_r):
    """(N, r, K, jac): node radii, K_i (= (dr/di)^2 on the logarithmic grid, h^2 on the uniform one) and dr/di, as the engine builds them."""
    N = 2 ** levels + 1
    i = np.arange(N, dtype=np.float64)
    if delta == 0.0:
        h = max_r / (N - 1)
        r = (max_r * i) / (N - 1)
        return N, r, np.full(N, h * h), np.full(N, h)
    rp = max_r / (np.exp((N - 1) * delta) - 1.0)
    ex = np.exp(i * delta)
    return N, rp * (ex - 1.0), (rp * delta * ex) ** 2, rp * delta * ex


def nearest_node(r, r_c):
    """The node the engine uses for r_c (r_2 <= r_c <= r_(N-2)): the nearest one, ties to the inner node."""
    N = len(r)
    hi = int(np.searchsorted(r[2:N - 1], r_c, side="left")) + 2
    return hi - 1 if hi > 2 and r_c - r[hi - 1] <= r[hi] - r_c else hi


def simpson_weights(n):
    """Weights of nodes 0..n: Simpson 1/3 on 0..m (m = n, or n - 3 when n is odd) plus the 3/8 rule on m..n."""
    m = n if n % 2 == 0 else n - 3
    w = np.zeros(n + 1)
    if m > 0:
        w[1:m:2] = 4.0 / 3.0
        w[2:m - 1:2] = 2.0 / 3.0
        w[0] += 1.0 / 3.0
        w[m] += 1.0 / 3.0
    if n % 2:
        w[m:m + 4] += np.array([3.0, 9.0, 9.0, 3.0]) / 8.0
    return w


def log_derivative(V, levels, delta, max_r, l, r_c, E):
    """D, u, du, nodes ([n_energies] each) and the radius used, for one channel (V [N], l, r_c) at the energies E."""
    N, r, K, jac = grid(levels, delta, max_r)
    n = nearest_node(r, r_c)
    E = np.atleast_1d(np.asarray(E, dtype=np.float64))
    V = np.asarray(V, dtype=np.float64)
    rr = np.where(r > 0, r, 1.0)
    g0 = (2.0 * K * V + np.where(r > 0, K * l * (l + 1) / rr ** 2, 0.0) + delta * delta / 4.0) / 12.0     # g at E = 0
    gE = K / 6.0                                                                                         # -dg/dE
    wt = simpson_weights(n)
    uniform = delta == 0.0
    y = np.full(E.shape, (max_r / (N - 1)) ** (l + 1) if uniform else r[1] ** (l + 1) * np.exp(-0.5 * delta))
    g = g0[1] - E * gE[1]
    wprev, w = np.zeros_like(y), (1.0 - g) * y
    s = wt[1] * y * y * (1.0 if uniform else np.exp(delta)) * jac[1]
    positive = np.ones(E.shape, bool)
    nodes = np.zeros(E.shape, np.int64)
    bad = np.zeros(E.shape, bool)
    ys, gs = {1: y}, {1: g}
    for i in range(2, n + 2):
        gi = g0[i] - E * gE[i]
        wn = 2.0 * w - wprev + 12.0 * g * y
        wprev, w = w, wn
        d = 1.0 - gi
        bad |= ~(d > 0)
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            y = wn / d
        g = gi
        if i <= n:
            flip = np.where(positive, y < 0, y > 0)
            nodes += flip
            positive ^= flip
            s = s + wt[i] * y * y * (1.0 if uniform else np.exp(delta * i)) * jac[i]
            big = np.abs(y) > _BIG
            if big.any():
                for a in (y, w, wprev):
                    a[big] *= _DOWN
                s[big] *= _DOWN * _DOWN
                for k in ys:
                    ys[k] = np.where(big, ys[k] * _DOWN, ys[k])
        if i >= n - 1:
            ys[i], gs[i] = y, g
    dy = ((1.0 - 2.0 * gs[n + 1]) * ys[n + 1] - (1.0 - 2.0 * gs[n - 1]) * ys[n - 1]) / 2.0
    if uniform:
        h = max_r / (N - 1)
        uc, du = ys[n], dy / h
    else:
        rp = max_r / (np.exp((N - 1) * delta) - 1.0)
        uc = ys[n] * np.exp(0.5 * delta * n)
        du = np.exp(-0.5 * delta * n) * (dy + 0.5 * delta * ys[n]) / (rp * delta)
    with np.errstate(invalid="ignore", divide="ignore"):
        norm = np.sqrt(s)
        D, u, du = du / uc, uc / norm, du / norm
    nodes = np.where(bad, -1, nodes)
    D, u, du = (np.where(bad, np.nan, x) for x in (D, u, du))
    return D, u, du, nodes, r[n]


def phase(D, nodes, r_c):
    """pi nodes - atan(r_c D): continuous across the poles of D and increasing in E."""
    return np.pi * nodes - np.arctan(r_c * D)
