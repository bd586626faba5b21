// Host-side occupation rules (integer logic, runs once per atom).
// Replaces AufbauPrinciple::GetSubshells (reference DFTAtom/AufbauPrinciple.h:36-75, exceptions :101-117,
// :129-142) + the driver's sort by (n,l) (DFTAtom.cpp:367) and DFTAtom::InitializeLevels (DFTAtom.cpp:611-638).
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>
#include "internal.h"

namespace dft {

namespace {

struct Shell { int n0, l, occ; };

// f-block / Lr adjustments.  The reference applies the same adjustment twice around the "electrons left"
// clamp (AufbauPrinciple.h:53,59); the transition-metal rules (:78-99) exist there but are never invoked,
// so Cr comes out 3d4 4s2 — reproduced on purpose.
int adjust(int occ, int Z, int n0, int l)
{
    if (l == 3) {
        const bool la_ce_gd = (Z == 57 || Z == 58 || Z == 64);
        if (la_ce_gd && n0 == 3) return occ - 1;
        if (n0 == 4) {
            if (Z == 89 || Z == 90) return 0;
            if (Z == 91 || Z == 92 || Z == 93 || Z == 96) return occ - 1;
        }
    } else if (Z == 103 && n0 == 5 && l == 2) {
        return 0;
    }
    return occ;
}

std::vector<Shell> fill(int Z)
{
    std::vector<Shell> v;
    int placed = 0;
    for (int sum = 0; sum < 10 && placed != Z; ++sum)
        for (int n0 = 0; n0 <= sum && placed != Z; ++n0) {
            const int l = sum - n0;
            if (l > n0) continue;
            int occ = adjust(2 * (2 * l + 1), Z, n0, l);
            occ = std::min(occ, Z - placed);
            occ = adjust(occ, Z, n0, l);
            if (occ > 0) { v.push_back({ n0, l, occ }); placed += occ; }
        }
    std::sort(v.begin(), v.end(), [](const Shell& a, const Shell& b) { return a.n0 != b.n0 ? a.n0 < b.n0 : a.l < b.l; });
    return v;
}

dftatom_level to_level(const Shell& s)
{
    dftatom_level L;
    L.n = s.n0 + 1; L.l = s.l; L.occ = s.occ; L.nodes = s.n0 - s.l; L.E = 0.;
    return L;
}

}  // namespace

int aufbau(int Z, dftatom_level* out, int max_out)
{
    if (Z < 1 || Z > 118) return DFTATOM_E_BAD_OPTION;
    const std::vector<Shell> v = fill(Z);
    if ((int)v.size() > max_out) return DFTATOM_E_ARG;
    for (size_t k = 0; k < v.size(); ++k) out[k] = to_level(v[k]);
    return (int)v.size();
}

int split_spin(int Z, dftatom_level* a, int* na, dftatom_level* b, int* nb, int* ea, int* eb)
{
    dftatom_level all[DFTATOM_MAX_LEVELS];
    const int n = aufbau(Z, all, DFTATOM_MAX_LEVELS);
    if (n < 0) return n;
    int ka = 0, kb = 0, n_alpha = 0;
    for (int k = 0; k < n; ++k) {
        const int cap = 2 * all[k].l + 1;                 // getMaxNrAlphaElectrons, AufbauPrinciple.h:26-29
        const int up = std::min(all[k].occ, cap);
        a[ka] = all[k]; a[ka].occ = up; ++ka;
        n_alpha += up;
        if (all[k].occ - up > 0) { b[kb] = all[k]; b[kb].occ = all[k].occ - up; ++kb; }
    }
    *na = ka; *nb = kb; *ea = n_alpha; *eb = Z - n_alpha;
    return 0;
}

// The reference's configuration ionised by `charge` electrons (rule and examples: dftatom_config_aufbau in dftatom_b200.h)
int config_aufbau(int Z, int method, double charge, dftatom_config* out)
{
    if (!out) return DFTATOM_E_ARG;
    if (Z < 1 || Z > 118 || !(charge >= -2. && charge < (double)Z) || method < 0 || method > 3) {
        set_error("config_aufbau: Z = " + std::to_string(Z) + ", charge = " + std::to_string(charge) + " (needs 1 <= Z <= 118, -2 <= charge < Z)");
        return DFTATOM_E_BAD_OPTION;
    }
    const std::vector<Shell> v = fill(Z);          // (n, l) order
    std::vector<double> occ(v.size());
    for (size_t k = 0; k < v.size(); ++k) occ[k] = v[k].occ;
    std::vector<Shell> shells = v;
    if (charge > 0.) {
        double left = charge;
        while (left > 0.) {                         // the occupied subshell of largest n, then largest l: the last one in (n, l) order
            size_t k = shells.size();
            while (k > 0 && !(occ[k - 1] > 0.)) --k;
            if (k == 0) break;
            const double take = std::min(occ[k - 1], left);
            occ[k - 1] -= take; left -= take;
        }
    } else if (charge < 0.) {
        // every subshell in the filling order of fill() (Madelung), gaining from the first one that is not full
        std::vector<Shell> order;
        for (int sum = 0; sum < 10; ++sum)
            for (int n0 = 0; n0 <= sum; ++n0) { const int l = sum - n0; if (l <= n0 && l <= 3) order.push_back({ n0, l, 0 }); }
        double left = -charge;
        bool started = false;
        for (const Shell& o : order) {
            if (!(left > 0.)) break;
            size_t k = 0;
            while (k < shells.size() && !(shells[k].n0 == o.n0 && shells[k].l == o.l)) ++k;
            const double cap = 2. * (2 * o.l + 1), have = k < shells.size() ? occ[k] : 0.;
            if (!started && have >= cap) continue;
            started = true;
            const double add = std::min(cap - have, left);
            if (add <= 0.) continue;
            if (k == shells.size()) { shells.push_back(o); occ.push_back(0.); }
            occ[k] += add; left -= add;
        }
    }
    std::vector<size_t> idx;
    for (size_t k = 0; k < shells.size(); ++k) if (occ[k] > 0.) idx.push_back(k);
    std::sort(idx.begin(), idx.end(), [&](size_t x, size_t y) { return shells[x].n0 != shells[y].n0 ? shells[x].n0 < shells[y].n0 : shells[x].l < shells[y].l; });
    int m = 0;
    const bool lsda = method & 1;
    for (int spin = 0; spin < (lsda ? 2 : 1); ++spin)
        for (size_t k : idx) {
            const double cap = 2 * shells[k].l + 1;
            const double o = !lsda ? occ[k] : spin == 0 ? std::min(occ[k], cap) : occ[k] - std::min(occ[k], cap);
            if (spin == 1 && !(o > 0.)) continue;
            out->orb[m++] = dftatom_occupation{ shells[k].n0 + 1, shells[k].l, spin, o };
        }
    out->n_orbitals = m;
    return 0;
}

int atom_levels(int atom, const dftatom_options& o, const dftatom_config* cfg, AtomLevels* out, double z_val)
{
    const bool lsda = o.method & 1;
    for (int s = 0; s < 2; ++s) { out->lev[s].clear(); out->occ[s].clear(); }
    if (!cfg || cfg->n_orbitals == 0) {
        dftatom_level la[DFTATOM_MAX_LEVELS], lb[DFTATOM_MAX_LEVELS];
        int na = 0, nb = 0, ea = o.Z, eb = 0;
        if (lsda) { int rc = split_spin(o.Z, la, &na, lb, &nb, &ea, &eb); if (rc) return rc; }
        else { na = aufbau(o.Z, la, DFTATOM_MAX_LEVELS); if (na < 0) return na; }
        out->lev[0].assign(la, la + na); out->lev[1].assign(lb, lb + nb);
        for (int s = 0; s < 2; ++s) for (const auto& x : out->lev[s]) out->occ[s].push_back(x.occ);
        out->n_el[0] = ea; out->n_el[1] = eb;
        return 0;
    }
    auto bad = [&](int k, const std::string& why) {
        std::string e = "atom " + std::to_string(atom) + (z_val > 0. ? " (z_val = " + std::to_string(z_val) : " (Z = " + std::to_string(o.Z)) + "): configuration";
        if (k >= 0) {
            const dftatom_occupation& x = cfg->orb[k];
            e += " entry " + std::to_string(k) + " (n = " + std::to_string(x.n) + ", l = " + std::to_string(x.l) + ", spin = " + std::to_string(x.spin)
                 + ", occ = " + std::to_string(x.occ) + ")";
        }
        set_error(e + ": " + why);
        return DFTATOM_E_BAD_OPTION;
    };
    if (cfg->n_orbitals < 0 || cfg->n_orbitals > 2 * DFTATOM_MAX_LEVELS) return bad(-1, "n_orbitals must be 0 .. 2 DFTATOM_MAX_LEVELS");
    std::vector<int> ord[2];
    double q = 0.;
    for (int k = 0; k < cfg->n_orbitals; ++k) {
        const dftatom_occupation& x = cfg->orb[k];
        if (x.n < 1 || x.n > 8) return bad(k, "needs 1 <= n <= 8");
        if (x.l < 0 || x.l > std::min(3, x.n - 1)) return bad(k, "needs 0 <= l <= min(3, n - 1)");
        if (x.spin != 0 && !(lsda && x.spin == 1)) return bad(k, lsda ? "spin must be 0 (alpha) or 1 (beta)" : "spin must be 0 for LDA");
        const double cap = (lsda ? 1. : 2.) * (2 * x.l + 1);
        if (!std::isfinite(x.occ)) return bad(k, "occupation is not finite");
        if (!(x.occ >= 0. && x.occ <= cap)) return bad(k, "needs 0 <= occ <= " + std::to_string((int)cap));
        for (int j = 0; j < k; ++j)
            if (cfg->orb[j].n == x.n && cfg->orb[j].l == x.l && cfg->orb[j].spin == x.spin) return bad(k, "duplicates entry " + std::to_string(j));
        ord[x.spin].push_back(k);
        q += x.occ;
    }
    if (ord[0].empty()) return bad(-1, "has no alpha (spin 0) entry");
    for (int s = 0; s < 2; ++s)
        if ((int)ord[s].size() > DFTATOM_MAX_LEVELS) return bad(-1, "more than DFTATOM_MAX_LEVELS entries of one spin");
    if (z_val > 0. ? !(q > 0. && q <= z_val + 2.) : !(q > 0. && q <= o.Z + 2.))
        return bad(-1, "electron count " + std::to_string(q) + (z_val > 0. ? " outside (0, z_val + 2]" : " outside (0, Z + 2]"));
    for (int s = 0; s < 2; ++s) {
        std::stable_sort(ord[s].begin(), ord[s].end(), [&](int x, int y) {
            const dftatom_occupation &a = cfg->orb[x], &b = cfg->orb[y];
            return a.n != b.n ? a.n < b.n : a.l < b.l;
        });
        double ne = 0.;
        for (int k : ord[s]) {
            const dftatom_occupation& x = cfg->orb[k];
            dftatom_level L;
            L.n = x.n; L.l = x.l; L.occ = (int)std::lround(x.occ); L.nodes = x.n - x.l - 1; L.E = 0.;
            out->lev[s].push_back(L); out->occ[s].push_back(x.occ);
            ne += x.occ;
        }
        out->n_el[s] = ne;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------
// Sharding of a batch of independent atoms over G GPUs (SURVEY 8e: one process per GPU, no collective).
// Cost of an atom = (spin) orbitals x expected SCF steps.  Which atoms take 60-150 steps instead of ~35 is physics, not Z: the
// NODELESS compact d / f shells (3d, 4f: n = l + 1) slosh under linear mixing when they are nearly full (Cu, Zn: 89 / 69 steps,
// Ho .. Yb: 77 .. 100 steps of the reference's sweep, SURVEY B.1; their 4d / 5d / 5f counterparts do not).  Only used to balance
// shards - a wrong estimate costs time, never results.
// ---------------------------------------------------------------------------------------------------------
double estimate_cost(int Z, int method)
{
    if (Z < 1 || Z > 118) return 0.;
    const std::vector<Shell> v = fill(Z);
    int n_orb = 0;
    for (const Shell& s : v) n_orb += (method && s.occ > 2 * s.l + 1) ? 2 : 1;
    // the subshells in Madelung (filling) order: the one filled last, and the one before it
    std::vector<const Shell*> order;
    for (const Shell& s : v) order.push_back(&s);
    std::sort(order.begin(), order.end(), [](const Shell* a, const Shell* b) { return a->n0 + a->l != b->n0 + b->l ? a->n0 + a->l < b->n0 + b->l : a->n0 < b->n0; });
    double steps = method ? 50. : 36.;
    for (size_t q = order.size() >= 2 ? order.size() - 2 : 0; q < order.size(); ++q) {
        const Shell& s = *order[q];
        if (s.l < 1 || s.n0 != s.l) continue;                   // nodeless: n = l + 1 (n0 is 0-based)
        const bool is_last = q + 1 == order.size();
        const double x = (double)s.occ / (double)(2 * (2 * s.l + 1));
        if (x > 0.7) steps += (method ? 100. : 65.) * (x - 0.7) / 0.3 * (s.l >= 2 ? 1. : 0.2) * (is_last ? 1. : 0.4);
    }
    return (double)n_orb * steps;
}

// longest-processing-time-first: atoms in order of decreasing cost, each to the least loaded rank; deterministic
int partition_atoms(const int* Z, const int* method, int n, int n_ranks, int* rank_of)
{
    if (!Z || !rank_of || n < 0 || n_ranks < 1) return DFTATOM_E_ARG;
    std::vector<double> cost(n);
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) { cost[i] = estimate_cost(Z[i], method ? method[i] : 0); order[i] = i; }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    std::vector<double> load(n_ranks, 0.);
    for (int i : order) {
        int r = 0;
        for (int q = 1; q < n_ranks; ++q) if (load[q] < load[r]) r = q;
        rank_of[i] = r;
        load[r] += cost[i];
    }
    return 0;
}

}  // namespace dft
