// dftatom — headless replacement of the reference's wxWidgets shell (DFTAtomApp / DFTAtomFrame / OptionsFrame).
// Flags carry the reference's Options fields with the same defaults (Options.cpp:6) and dialog ranges
// (OptionsFrame.cpp:46,152-173); the output is the text the reference's worker thread prints (DFTAtomFrame.cpp:185-198
// -> DFTAtom.cpp:358-490 / :857-1021).  All computation goes through the C ABI of include/dftatom_b200.h.
//
//   dftatom [--Z 18 | --Z 1-92 | --Z 21,22,57] [--levels 14] [--delta 0.0005] [--mixing 0.5] [--rmax 25]
//           [--method 0|1|lda|lsda] [--precision 6] [--json] [--quiet-steps] [--device 0] [--gpus N] [--ini DFTAtom.ini] [--radial DIR]
// --json: one record per atom (final energies, levels, and - unless --quiet-steps - every step at 17 digits)
// --gpus N: the batch is sharded over N GPUs, ONE PROCESS PER GPU (fork + exec of this binary with --device r and its share of the
//           atoms, longest-processing-time-first on dftatom_estimate_cost), no collective; the parent gathers the children's output
//           through pipes and prints it in the order of --Z, so the result is byte-identical to the 1-GPU run.
// --radial DIR: the converged radial state of every atom as a text table DIR/<index>_Z<Z>.tsv (index = position in --Z), one row per
//           grid node at 17 digits: r, rho per spin, V per spin, V_H, u(r) of every orbital (dftatom_solve_batch_radial).  With --gpus
//           every shard writes the files of its own atoms, named by their position in the whole --Z list.
// --charge Q: every atom of --Z is the reference's configuration ionised by Q electrons (dftatom_config_aufbau; fractional allowed,
//           < 0 = anion), e.g. --Z 1-92 --charge 1 for all cations.  --config "[Ne] 3s1 3p0": one atom (a single --Z) in that configuration
//           (subshells "2p4.5", LSDA also "2p3/1" = alpha / beta, cores [He] .. [Rn]; the same string form as dftatom_b200.parse_config).
//           Both are passed on to the shards of --gpus and select the rows of --radial.
// --logderiv DIR --rc R [--energies lo:hi:n]: logarithmic derivatives D_l(E) = u'(R) / u(R) of every atom's converged potential, l = 0..3
//           for each spin, at n energies from lo to hi (default -2:1:301), as a long table DIR/<index>_Z<Z>_logderiv.tsv with the columns
//           spin, l, E, D, nodes, phase = pi nodes - atan(r_c D), u, du at 17 digits (dftatom_log_derivatives; r_c = the grid node nearest
//           to R).  The potential is the one the radial export returns; --radial is not needed.  Works with --gpus, --charge and --config.
// --pseudo DIR --pseudo-rc Rs[,Rp,Rd,Rf]: Troullier-Martins pseudopotentials of every (LDA) atom (dftatom_tm_pseudize): for every l of the
//           atom's levels the level of largest n is the valence channel, at the radius given for that l (an l beyond the list takes the
//           last radius), and all channels of the atom are unscreened together.  DIR/<index>_Z<Z>_pseudo.tsv holds one "#" line per
//           channel (l n eps occ r_c status c0 .. c12) and the columns r, V_ion per l, V_scr per l, u per l and rho_val at 17 digits.
//           With --logderiv DIR2 --rc R (R >= every pseudo radius) also DIR2/<index>_Z<Z>_pseudo_logderiv.tsv: the logarithmic
//           derivatives of the V_scr channels at the --energies, in the columns of the all-electron table (spin 0).  LSDA atoms are an
//           error; works with --gpus, --charge and --config and does not need --radial.
// --pseudo-local L: with --pseudo, the Kleinman-Bylander form of every atom's channels with the channel of l = L as the local potential
//           (dftatom_kb_form): one "# kb" line per channel (l E_KB cos eps_loc0 eps_loc1 ghost status) after the channel lines and one
//           beta column per channel after rho_val.  With --logderiv also DIR2/<index>_Z<Z>_pseudo_kb_logderiv.tsv, the KB logarithmic
//           derivatives (dftatom_kb_log_derivatives) in the layout of the pseudo table.  An atom without a channel of l = L is an error.
// --pseudo-test "3s1 3p3;3s2 3p1": with --pseudo and a single --Z, the transferability test of its pseudopotentials: the pseudo-atom
//           (dftatom_solve_pseudo_batch) in the reference valence configuration and in each listed one, and the all-electron atom in core +
//           each of them (the core: every reference entry whose n is below its channel's reference n, or whose l has no channel).
//           DIR/<index>_Z<Z>_pseudo_test.tsv: one row per configuration (config Q E_AE E_PS dE_AE dE_PS dE_PS-dE_AE status_AE status_PS;
//           dE against the reference configuration), then one "# level" line per level (config n l spin occ eps_AE eps_PS).
// --pseudo-core R: with --pseudo, the nonlinear core correction: the core density of the atom's other (core) levels, its Louie-Froyen-
//           Cohen partial core at radius R (0 = the full core, dftatom_partial_core), and the unscreening with it
//           (dftatom_tm_pseudize_core); --pseudo-test then solves the pseudo-atoms with it (dftatom_solve_pseudo_batch_core).  The pseudo
//           table gains a "# core" line (r_pc i_pc A B n_core n_pc status) after the channel and kb lines and the columns rho_core and
//           rho_pc after the others.
#include <algorithm>
#include <cmath>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>
#include <cerrno>
#include <sys/stat.h>
#include <sys/types.h>
#include <sys/wait.h>
#include <unistd.h>
#include "../../include/dftatom_b200.h"

static const char kOrb[] = "spdf";

static std::vector<int> parse_z(const std::string& s)
{
    std::vector<int> out;
    size_t pos = 0;
    while (pos < s.size()) {
        size_t comma = s.find(',', pos);
        std::string tok = s.substr(pos, comma == std::string::npos ? std::string::npos : comma - pos);
        size_t dash = tok.find('-', 1);
        if (dash != std::string::npos) {
            int a = std::atoi(tok.substr(0, dash).c_str()), b = std::atoi(tok.substr(dash + 1).c_str());
            for (int z = a; z <= b; ++z) out.push_back(z);
        } else if (!tok.empty()) out.push_back(std::atoi(tok.c_str()));
        if (comma == std::string::npos) break;
        pos = comma + 1;
    }
    return out;
}

// reads the keys the reference persists with wxFileConfig (Options.cpp:42-49): Z, MultigridLevels, MaxR, deltaGrid, alpha, Method
static void read_ini(const char* path, dftatom_options& o)
{
    std::ifstream f(path);
    std::string line;
    while (std::getline(f, line)) {
        size_t eq = line.find('=');
        if (eq == std::string::npos) continue;
        std::string k = line.substr(0, eq), v = line.substr(eq + 1);
        while (!k.empty() && (k.back() == ' ' || k.back() == '\t')) k.pop_back();
        while (!k.empty() && (k[0] == '/' || k[0] == ' ')) k.erase(0, 1);
        if (k == "Z") o.Z = std::atoi(v.c_str());
        else if (k == "MultigridLevels") o.levels = std::atoi(v.c_str());
        else if (k == "MaxR") o.max_r = std::atof(v.c_str());
        else if (k == "deltaGrid") o.delta = std::atof(v.c_str());
        else if (k == "alpha") o.mixing = std::atof(v.c_str());
        else if (k == "Method") o.method = std::atoi(v.c_str());
    }
}

// the exact occupation of a level: a configured atom's entry with the same (n, l, spin) (dftatom_level.occ holds it rounded)
static double exact_occ(const dftatom_level& L, int spin, const dftatom_config* cfg)
{
    for (int q = 0; cfg && q < cfg->n_orbitals; ++q)
        if (cfg->orb[q].n == L.n && cfg->orb[q].l == L.l && cfg->orb[q].spin == spin) return cfg->orb[q].occ;
    return L.occ;
}

// occupations with %g: integers print as the reference prints them
static void print_conf(const dftatom_level* lv, int n, int spin, const dftatom_config* cfg)
{
    for (int k = 0; k < n; ++k) std::printf("%d%c%g ", lv[k].n, kOrb[lv[k].l], exact_occ(lv[k], spin, cfg));
}

// the string form of a configuration (dftatom_b200.parse_config): returns false with a message on stderr
static bool parse_config(const std::string& s, int method, dftatom_config* out)
{
    static const struct { const char* sym; int Z; } kCores[] = { { "[He]", 2 }, { "[Ne]", 10 }, { "[Ar]", 18 }, { "[Kr]", 36 }, { "[Xe]", 54 }, { "[Rn]", 86 } };
    const bool lsda = method & 1;
    std::vector<dftatom_occupation> v;
    auto drop = [&](int n, int l) { v.erase(std::remove_if(v.begin(), v.end(), [&](const dftatom_occupation& e) { return e.n == n && e.l == l; }), v.end()); };
    size_t pos = 0;
    while (pos < s.size()) {
        while (pos < s.size() && std::isspace((unsigned char)s[pos])) ++pos;
        if (pos >= s.size()) break;
        size_t end = pos;
        while (end < s.size() && !std::isspace((unsigned char)s[end])) ++end;
        const std::string tok = s.substr(pos, end - pos);
        pos = end;
        int coreZ = 0;
        for (const auto& c : kCores) if (tok == c.sym) coreZ = c.Z;
        if (coreZ) {
            dftatom_config core;
            if (dftatom_config_aufbau(coreZ, method, 0., &core) != DFTATOM_OK) return false;
            for (int q = 0; q < core.n_orbitals; ++q) drop(core.orb[q].n, core.orb[q].l);
            v.insert(v.end(), core.orb, core.orb + core.n_orbitals);
            continue;
        }
        const char* p = tok.c_str();
        const char* lp = tok.size() >= 3 && std::isdigit((unsigned char)p[0]) ? std::strchr(kOrb, p[1]) : nullptr;
        char* e1 = nullptr;
        const double a = lp && p[1] ? std::strtod(p + 2, &e1) : 0.;
        double b = -1.;
        bool ok = lp && e1 && e1 != p + 2;
        if (ok && *e1 == '/') { char* e2 = nullptr; b = std::strtod(e1 + 1, &e2); ok = lsda && e2 != e1 + 1 && *e2 == 0; }
        else ok = ok && *e1 == 0;
        if (!ok) { std::fprintf(stderr, "dftatom: --config: cannot read '%s' (expected e.g. 3d10, 2p4.5, [Ar]%s)\n", tok.c_str(), lsda ? ", 2p3/1" : ""); return false; }
        const int n = p[0] - '0', l = (int)(lp - kOrb);
        drop(n, l);
        if (b >= 0.) { v.push_back({ n, l, 0, a }); v.push_back({ n, l, 1, b }); }
        else if (lsda) { const double up = std::min(a, 2. * l + 1.); v.push_back({ n, l, 0, up }); if (a - up > 0.) v.push_back({ n, l, 1, a - up }); }
        else v.push_back({ n, l, 0, a });
    }
    if (v.size() > 2 * DFTATOM_MAX_LEVELS) { std::fprintf(stderr, "dftatom: --config: too many subshells\n"); return false; }
    out->n_orbitals = (int)v.size();
    std::copy(v.begin(), v.end(), out->orb);
    return true;
}

// --gpus N: one child process per GPU (CUDA is only ever initialised in the children), each solving its shard as one batch.
static int run_sharded(const char* self, const std::vector<int>& zs, int method, int gpus, const std::vector<std::string>& pass, bool json)
{
    const int n = (int)zs.size();
    std::vector<int> meth(n, method), rank_of(n, 0);
    if (dftatom_partition(zs.data(), meth.data(), n, gpus, rank_of.data()) != DFTATOM_OK) { std::fprintf(stderr, "dftatom: bad --gpus\n"); return 2; }
    struct Child { pid_t pid; int fd; std::vector<int> atoms; std::string out; };
    std::vector<Child> ch(gpus);
    for (int r = 0; r < gpus; ++r) {
        Child& c = ch[r];
        c.pid = -1; c.fd = -1;
        for (int i = 0; i < n; ++i) if (rank_of[i] == r) c.atoms.push_back(i);
        if (c.atoms.empty()) continue;
        std::string zlist;
        for (size_t q = 0; q < c.atoms.size(); ++q) zlist += (q ? "," : "") + std::to_string(zs[c.atoms[q]]);
        int pfd[2];
        if (pipe(pfd) != 0) { std::perror("pipe"); return 1; }
        c.pid = fork();
        if (c.pid < 0) { std::perror("fork"); return 1; }
        if (c.pid == 0) {
            dup2(pfd[1], 1); close(pfd[0]); close(pfd[1]);
            // shard r runs on GPU r; DFTATOM_SHARD_DEVICES="0,0" (a comma list, used round-robin) overrides the mapping, e.g. to run two
            // shards on one GPU
            int dev = r;
            if (const char* map = std::getenv("DFTATOM_SHARD_DEVICES")) { const std::vector<int> ids = parse_z(map); if (!ids.empty()) dev = ids[r % ids.size()]; }
            std::string ilist;
            for (size_t q = 0; q < c.atoms.size(); ++q) ilist += (q ? "," : "") + std::to_string(c.atoms[q]);
            std::vector<std::string> args = { self, "--framed", "--device", std::to_string(dev), "--Z", zlist, "--atom-index", ilist };
            args.insert(args.end(), pass.begin(), pass.end());
            std::vector<char*> av;
            for (auto& a : args) av.push_back(const_cast<char*>(a.c_str()));
            av.push_back(nullptr);
            execv(self, av.data());
            std::perror("execv");
            _exit(127);
        }
        close(pfd[1]);
        c.fd = pfd[0];
    }
    int rc = 0;
    for (Child& c : ch) {                   // the children run concurrently; their (small) outputs are drained one after the other
        if (c.pid < 0) continue;
        char buf[1 << 16];
        ssize_t k;
        while ((k = read(c.fd, buf, sizeof buf)) > 0) c.out.append(buf, (size_t)k);
        close(c.fd);
        int st = 0;
        waitpid(c.pid, &st, 0);
        if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) rc = 1;
    }
    if (rc) { std::fprintf(stderr, "dftatom: a shard failed\n"); return rc; }
    // gather on the host: frames "\x1e<k>\n<text>" of every child, re-ordered to the order of --Z
    std::vector<std::string> rec(n);
    for (Child& c : ch) {
        size_t pos = 0;
        while ((pos = c.out.find('\x1e', pos)) != std::string::npos) {
            const size_t nl = c.out.find('\n', pos);
            const int k = std::atoi(c.out.substr(pos + 1, nl - pos - 1).c_str());
            size_t end = c.out.find('\x1e', nl);
            if (end == std::string::npos) end = c.out.size();
            if (k >= 0 && k < (int)c.atoms.size()) rec[c.atoms[k]] = c.out.substr(nl + 1, end - nl - 1);
            pos = end;
        }
    }
    if (json) std::printf("[");
    for (int i = 0; i < n; ++i) std::printf("%s%s", (json && i) ? "," : "", rec[i].c_str());
    if (json) std::printf("]\n");
    return 0;
}

// --radial: one table per atom, columns r | rho per spin | V per spin | V_H | u of every orbital (headed like the report: "2p"; LSDA "alpha 2p")
static int write_radial(const std::string& dir, int index, const dftatom_options& o, const dftatom_result& R, int N, const double* r,
                        const double* rho, const double* v, const double* vh, const double* orb)
{
    const std::string path = dir + "/" + std::to_string(index) + "_Z" + std::to_string(o.Z) + ".tsv";
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) { std::perror(path.c_str()); return 1; }
    const int ns = R.n_spin;
    static const char* const kSpin[2] = { "alpha", "beta" };
    std::fprintf(f, "# r");
    for (const char* q : { "rho", "V" })
        for (int s = 0; s < ns; ++s) std::fprintf(f, ns == 2 ? "\t%s %s" : "\t%s", q, kSpin[s]);
    std::fprintf(f, "\tV_H");
    int n_orb = 0;
    for (int s = 0; s < ns; ++s)
        for (int k = 0; k < R.n_levels[s]; ++k, ++n_orb) {
            if (ns == 2) std::fprintf(f, "\t%s %d%c", kSpin[s], R.levels[s][k].n, kOrb[R.levels[s][k].l]);
            else std::fprintf(f, "\t%d%c", R.levels[s][k].n, kOrb[R.levels[s][k].l]);
        }
    std::fprintf(f, "\n");
    for (int i = 0; i < N; ++i) {
        std::fprintf(f, "%.17g", r[i]);
        for (int s = 0; s < ns; ++s) std::fprintf(f, "\t%.17g", rho[(size_t)s * N + i]);
        for (int s = 0; s < ns; ++s) std::fprintf(f, "\t%.17g", v[(size_t)s * N + i]);
        std::fprintf(f, "\t%.17g", vh[i]);
        for (int k = 0; k < n_orb; ++k) std::fprintf(f, "\t%.17g", orb[(size_t)k * N + i]);
        std::fprintf(f, "\n");
    }
    const bool bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", path.c_str()); return 1; }
    return 0;
}

// --logderiv: channels l = 0..3 of every spin on the atom's converged V (rows of dftatom_radial.v), one long table
static int write_logderiv(dftatom_ctx* ctx, const std::string& dir, int index, const dftatom_options& o, int n_spin, const double* v,
                          double rc, const std::vector<double>& E)
{
    const int nc = 4 * n_spin, ne = (int)E.size();
    std::vector<int> pot(nc), l(nc);
    std::vector<double> rcs(nc, rc), used(nc);
    for (int c = 0; c < nc; ++c) { pot[c] = c / 4; l[c] = c % 4; }
    std::vector<dftatom_logderiv> out((size_t)nc * ne);
    if (dftatom_log_derivatives(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, v, n_spin, pot.data(), l.data(), rcs.data(), nc, E.data(), ne,
                                out.data(), used.data()) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --logderiv Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    const std::string path = dir + "/" + std::to_string(index) + "_Z" + std::to_string(o.Z) + "_logderiv.tsv";
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) { std::perror(path.c_str()); return 1; }
    std::fprintf(f, "# Z=%d method=%d r_c=%.17g\n# spin\tl\tE\tD\tnodes\tphase\tu\tdu\n", o.Z, o.method, used[0]);
    for (int c = 0; c < nc; ++c)
        for (int k = 0; k < ne; ++k) {
            const dftatom_logderiv& q = out[(size_t)c * ne + k];
            const double phase = q.nodes < 0 ? NAN : M_PI * q.nodes - std::atan(used[c] * q.D);
            std::fprintf(f, "%d\t%d\t%.17g\t%.17g\t%d\t%.17g\t%.17g\t%.17g\n", pot[c], l[c], E[k], q.D, q.nodes, phase, q.u, q.du);
        }
    const bool bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", path.c_str()); return 1; }
    return 0;
}

// --pseudo-test: the pseudo-atom of the channels ch (rows of v_ion) against the all-electron atom in the reference configuration and in
// every configuration of `tests`
static int pseudo_test(dftatom_ctx* ctx, const std::string& path, const dftatom_options& o, const dftatom_result& R, const dftatom_config* cfg,
                       const std::vector<dftatom_tm_channel>& ch, const std::vector<double>& v_ion, const std::vector<std::string>& tests,
                       const std::vector<double>& rho_pc)
{
    dftatom_pseudo_atom pa = {};
    for (int l = 0; l < 4; ++l) pa.row[l] = -1;
    for (size_t c = 0; c < ch.size(); ++c) { pa.row[ch[c].l] = (int)c; pa.n_ref[ch[c].l] = R.levels[0][ch[c].orbital].n; pa.z_val += ch[c].occ; }
    pa.mixing = o.mixing; pa.method = 0;
    // the reference configuration split into core and valence; its valence string
    dftatom_config core = {}, ref = {};
    std::string ref_str;
    for (int k = 0; k < R.n_levels[0]; ++k) {
        const dftatom_level& L = R.levels[0][k];
        const dftatom_occupation e = { L.n, L.l, 0, exact_occ(L, 0, cfg) };
        if (pa.row[L.l] < 0 || L.n < pa.n_ref[L.l]) core.orb[core.n_orbitals++] = e;
        else {
            ref.orb[ref.n_orbitals++] = e;
            char b[64];
            std::snprintf(b, sizeof b, "%s%d%c%.17g", ref_str.empty() ? "" : " ", L.n, kOrb[L.l], e.occ);
            ref_str += b;
        }
    }
    std::vector<std::string> names(1, ref_str);
    std::vector<dftatom_config> ps(1, ref);
    for (const std::string& t : tests) {
        dftatom_config c = {};
        if (!parse_config(t, 0, &c)) return 2;
        for (int k = 0; k < c.n_orbitals; ++k)
            if (pa.row[c.orb[k].l] < 0) {
                std::fprintf(stderr, "dftatom: --pseudo-test \"%s\": Z=%d has no pseudopotential channel with l = %d\n", t.c_str(), o.Z, c.orb[k].l);
                return 2;
            }
        names.push_back(t);
        ps.push_back(c);
    }
    const int n = (int)ps.size();
    std::vector<dftatom_config> ae(n, core);
    for (int q = 0; q < n; ++q)
        for (int k = 0; k < ps[q].n_orbitals; ++k) ae[q].orb[ae[q].n_orbitals++] = ps[q].orb[k];
    std::vector<dftatom_pseudo_atom> pas(n, pa);
    std::vector<dftatom_options> opts(n, o);
    std::vector<dftatom_result> r_ps(n), r_ae(n);
    const std::vector<int> pc_row(n, 0);          // with --pseudo-core every pseudo-atom takes the one partial core row
    if (dftatom_solve_pseudo_batch_core(ctx, o.levels, o.delta, o.max_r, v_ion.data(), (int)ch.size(), pas.data(), ps.data(), n, r_ps.data(), nullptr, 0,
                                        nullptr, rho_pc.empty() ? nullptr : rho_pc.data(), 1, rho_pc.empty() ? nullptr : pc_row.data()) != DFTATOM_OK ||
        dftatom_solve_batch_config(ctx, opts.data(), ae.data(), n, r_ae.data(), nullptr, 0, nullptr) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --pseudo-test Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) { std::perror(path.c_str()); return 1; }
    std::fprintf(f, "# Z=%d method=%d pseudo-atom test; dE against the reference configuration (row 1)\n", o.Z, o.method);
    std::fprintf(f, "# config\tQ\tE_AE\tE_PS\tdE_AE\tdE_PS\tdE_PS-dE_AE\tstatus_AE\tstatus_PS\n");
    for (int q = 0; q < n; ++q) {
        double Q = 0.;
        for (int k = 0; k < ps[q].n_orbitals; ++k) Q += ps[q].orb[k].occ;
        const double dae = r_ae[q].Etotal - r_ae[0].Etotal, dps = r_ps[q].Etotal - r_ps[0].Etotal;
        std::fprintf(f, "%s\t%.17g\t%.17g\t%.17g\t%.17g\t%.17g\t%.17g\t%d\t%d\n", names[q].c_str(), Q, r_ae[q].Etotal, r_ps[q].Etotal, dae, dps, dps - dae,
                     r_ae[q].status, r_ps[q].status);
    }
    std::fprintf(f, "# level\tconfig\tn\tl\tspin\tocc\teps_AE\teps_PS\n");
    for (int q = 0; q < n; ++q)
        for (int k = 0; k < r_ps[q].n_levels[0]; ++k) {
            const dftatom_level& L = r_ps[q].levels[0][k];
            double e_ae = NAN;
            for (int j = 0; j < r_ae[q].n_levels[0]; ++j)
                if (r_ae[q].levels[0][j].n == L.n && r_ae[q].levels[0][j].l == L.l) e_ae = r_ae[q].levels[0][j].E;
            std::fprintf(f, "# level\t%s\t%d\t%d\t%d\t%.17g\t%.17g\t%.17g\n", names[q].c_str(), L.n, L.l, 0, exact_occ(L, 0, &ps[q]), e_ae, L.E);
        }
    const bool bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", path.c_str()); return 1; }
    return 0;
}

// --pseudo: the valence channels of one LDA atom (largest n per l of its levels), pseudized and unscreened together; with --logderiv
// also the logarithmic derivatives of their V_scr rows at the all-electron table's radius and energies
static int write_pseudo(dftatom_ctx* ctx, const std::string& dir, const std::string& ld_dir, int index, const dftatom_options& o,
                        const dftatom_result& R, const dftatom_config* cfg, int N, const double* r, const double* v, const double* orb,
                        const std::vector<double>& rcs, double ld_rc, const std::vector<double>& E, int kb_loc,
                        const std::vector<std::string>& tests, double r_pc)
{
    int best[4] = { -1, -1, -1, -1 };
    for (int k = 0; k < R.n_levels[0]; ++k) {
        const dftatom_level& L = R.levels[0][k];
        if (best[L.l] < 0 || L.n > R.levels[0][best[L.l]].n) best[L.l] = k;
    }
    std::vector<dftatom_tm_channel> ch;
    for (int l = 0; l < 4; ++l) {
        if (best[l] < 0) continue;
        const dftatom_level& L = R.levels[0][best[l]];
        dftatom_tm_channel c = {};
        c.pot = 0; c.orbital = best[l]; c.l = l; c.eps = L.E; c.occ = exact_occ(L, 0, cfg);
        c.r_c = rcs[std::min<size_t>(l, rcs.size() - 1)];
        ch.push_back(c);
    }
    const int nc = (int)ch.size();
    std::vector<dftatom_tm_result> out(nc);
    std::vector<double> u_ps((size_t)nc * N), v_scr((size_t)nc * N), v_ion((size_t)nc * N), rho(N);
    // --pseudo-core: the partial core of the levels that are not valence channels
    const bool with_core = !std::isnan(r_pc);
    dftatom_pcc_result pcc = {};
    std::vector<double> rho_core(with_core ? N : 0), rho_pc(with_core ? N : 0);
    if (with_core) {
        std::vector<dftatom_core_orbital> core;
        for (int k = 0; k < R.n_levels[0]; ++k)
            if (k != best[R.levels[0][k].l]) core.push_back(dftatom_core_orbital{ 0, k, exact_occ(R.levels[0][k], 0, cfg) });
        if (dftatom_partial_core(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, orb, R.n_levels[0], core.data(), (int)core.size(), &r_pc, 1, &pcc,
                                 rho_core.data(), rho_pc.data()) != DFTATOM_OK) {
            std::fprintf(stderr, "dftatom: --pseudo-core Z=%d: %s\n", o.Z, dftatom_last_error());
            return 1;
        }
        if (pcc.status != 0) { std::fprintf(stderr, "dftatom: --pseudo-core Z=%d: the core density does not decrease at r_pc = %.17g\n", o.Z, pcc.r_pc); return 1; }
    }
    if (dftatom_tm_pseudize_core(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, v, 1, orb, R.n_levels[0], ch.data(), nc, out.data(), u_ps.data(),
                                 v_scr.data(), v_ion.data(), rho.data(), with_core ? rho_pc.data() : nullptr) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --pseudo Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    // --pseudo-local: the Kleinman-Bylander form with the channel of l = kb_loc as the local potential
    int loc = -1;
    for (int c = 0; c < nc; ++c) if (ch[c].l == kb_loc) loc = c;
    if (kb_loc >= 0 && loc < 0) { std::fprintf(stderr, "dftatom: --pseudo-local %d: Z=%d has no channel with l = %d\n", kb_loc, o.Z, kb_loc); return 1; }
    std::vector<dftatom_kb_channel> kch(loc >= 0 ? nc : 0);
    std::vector<dftatom_kb_result> kb(kch.size());
    std::vector<double> beta(kch.size() * (size_t)N);
    for (size_t c = 0; c < kch.size(); ++c) { kch[c] = dftatom_kb_channel{}; kch[c].row = (int)c; kch[c].loc = loc; kch[c].l = ch[c].l; kch[c].eps = ch[c].eps; }
    if (loc >= 0 && dftatom_kb_form(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, v_scr.data(), u_ps.data(), nc, kch.data(), nc, kb.data(),
                                    beta.data()) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --pseudo-local Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    const std::string stem = "/" + std::to_string(index) + "_Z" + std::to_string(o.Z) + "_pseudo";
    const std::string path = dir + stem + ".tsv";
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) { std::perror(path.c_str()); return 1; }
    std::fprintf(f, "# Z=%d method=%d channels: l n eps occ r_c status c0 c2 c4 c6 c8 c10 c12\n", o.Z, o.method);
    for (int c = 0; c < nc; ++c) {
        std::fprintf(f, "# %d\t%d\t%.17g\t%.17g\t%.17g\t%d", ch[c].l, R.levels[0][ch[c].orbital].n, ch[c].eps, ch[c].occ, out[c].r_c, out[c].status);
        for (int k = 0; k < 7; ++k) std::fprintf(f, "\t%.17g", out[c].c[k]);
        std::fprintf(f, "\n");
    }
    for (size_t c = 0; c < kb.size(); ++c)
        std::fprintf(f, "# kb\t%d\t%.17g\t%.17g\t%.17g\t%.17g\t%d\t%d\n", ch[c].l, kb[c].E_KB, kb[c].cos, kb[c].eps_loc[0], kb[c].eps_loc[1], kb[c].ghost,
                     kb[c].status);
    if (with_core)
        std::fprintf(f, "# core\t%.17g\t%d\t%.17g\t%.17g\t%.17g\t%.17g\t%d\n", pcc.r_pc, pcc.i_pc, pcc.A, pcc.B, pcc.n_core, pcc.n_pc, pcc.status);
    std::fprintf(f, "# r");
    for (const char* q : { "V_ion", "V_scr", "u" })
        for (int c = 0; c < nc; ++c) std::fprintf(f, "\t%s %c", q, kOrb[ch[c].l]);
    std::fprintf(f, "\trho_val");
    for (size_t c = 0; c < kb.size(); ++c) std::fprintf(f, "\tbeta %c", kOrb[ch[c].l]);
    if (with_core) std::fprintf(f, "\trho_core\trho_pc");
    std::fprintf(f, "\n");
    for (int i = 0; i < N; ++i) {
        std::fprintf(f, "%.17g", r[i]);
        for (const std::vector<double>* q : { &v_ion, &v_scr, &u_ps })
            for (int c = 0; c < nc; ++c) std::fprintf(f, "\t%.17g", (*q)[(size_t)c * N + i]);
        std::fprintf(f, "\t%.17g", rho[i]);
        for (size_t c = 0; c < kb.size(); ++c) std::fprintf(f, "\t%.17g", beta[c * N + i]);
        if (with_core) std::fprintf(f, "\t%.17g\t%.17g", rho_core[i], rho_pc[i]);
        std::fprintf(f, "\n");
    }
    bool bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", path.c_str()); return 1; }
    if (!tests.empty()) {
        const int rc_t = pseudo_test(ctx, dir + stem + "_test.tsv", o, R, cfg, ch, v_ion, tests, rho_pc);
        if (rc_t) return rc_t;
    }
    if (ld_dir.empty()) return 0;
    const int ne = (int)E.size();
    std::vector<int> pot(nc), l(nc);
    std::vector<double> lrc(nc, ld_rc), used(nc);
    for (int c = 0; c < nc; ++c) { pot[c] = c; l[c] = ch[c].l; }
    std::vector<dftatom_logderiv> ld((size_t)nc * ne);
    if (dftatom_log_derivatives(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, v_scr.data(), nc, pot.data(), l.data(), lrc.data(), nc, E.data(), ne,
                                ld.data(), used.data()) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --pseudo --logderiv Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    const std::string lpath = ld_dir + stem + "_logderiv.tsv";
    f = std::fopen(lpath.c_str(), "w");
    if (!f) { std::perror(lpath.c_str()); return 1; }
    std::fprintf(f, "# Z=%d method=%d r_c=%.17g V_scr\n# spin\tl\tE\tD\tnodes\tphase\tu\tdu\n", o.Z, o.method, used[0]);
    for (int c = 0; c < nc; ++c)
        for (int k = 0; k < ne; ++k) {
            const dftatom_logderiv& q = ld[(size_t)c * ne + k];
            const double phase = q.nodes < 0 ? NAN : M_PI * q.nodes - std::atan(used[c] * q.D);
            std::fprintf(f, "%d\t%d\t%.17g\t%.17g\t%d\t%.17g\t%.17g\t%.17g\n", 0, l[c], E[k], q.D, q.nodes, phase, q.u, q.du);
        }
    bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", lpath.c_str()); return 1; }
    if (loc < 0) return 0;
    // the KB channels at the same radius and energies: local potential V_scr of l = kb_loc, projector of every other channel
    std::vector<dftatom_kb_ld_channel> kl(nc);
    for (int c = 0; c < nc; ++c) {
        kl[c] = dftatom_kb_ld_channel{};
        kl[c].pot = loc; kl[c].proj = kb[c].status == 1 ? -1 : c; kl[c].l = ch[c].l; kl[c].E_KB = kb[c].status == 1 ? 0. : kb[c].E_KB; kl[c].r_c = ld_rc;
    }
    if (dftatom_kb_log_derivatives(ctx, o.levels, o.method >= 2 ? 0. : o.delta, o.max_r, v_scr.data(), nc, beta.data(), nc, kl.data(), nc, E.data(), ne,
                                   ld.data(), used.data()) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: --pseudo-local --logderiv Z=%d: %s\n", o.Z, dftatom_last_error());
        return 1;
    }
    const std::string kpath = ld_dir + stem + "_kb_logderiv.tsv";
    f = std::fopen(kpath.c_str(), "w");
    if (!f) { std::perror(kpath.c_str()); return 1; }
    std::fprintf(f, "# Z=%d method=%d r_c=%.17g KB l_loc=%d\n# spin\tl\tE\tD\tnodes\tphase\tu\tdu\n", o.Z, o.method, used[0], kb_loc);
    for (int c = 0; c < nc; ++c)
        for (int k = 0; k < ne; ++k) {
            const dftatom_logderiv& q = ld[(size_t)c * ne + k];
            const double phase = q.nodes < 0 ? NAN : M_PI * q.nodes - std::atan(used[c] * q.D);
            std::fprintf(f, "%d\t%d\t%.17g\t%.17g\t%d\t%.17g\t%.17g\t%.17g\n", 0, l[c], E[k], q.D, q.nodes, phase, q.u, q.du);
        }
    bad = std::ferror(f) != 0;
    if (std::fclose(f) != 0 || bad) { std::fprintf(stderr, "dftatom: write error on %s\n", kpath.c_str()); return 1; }
    return 0;
}

int main(int argc, char** argv)
{
    dftatom_options base = { 36, 12, 10.0, 0.001, 0.5, 0 };     // Options.cpp:6
    std::vector<int> zs, atom_index;                        // atom_index: positions of this shard's atoms in the parent's --Z list (--gpus children)
    std::string radial_dir, config_str, logderiv_dir, energies = "-2:1:301", pseudo_dir, pseudo_rc, pseudo_test;
    double charge = 0., rc = NAN, pseudo_core = NAN;
    int pseudo_local = -1;
    int precision = 6, device = 0, gpus = 1;
    bool json = false, quiet = false, framed = false;      // framed: child of --gpus (one frame per atom on stdout)
    std::vector<std::string> passthrough;                   // flags a --gpus parent hands to its children unchanged
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto next = [&]() -> const char* { if (i + 1 >= argc) { std::fprintf(stderr, "missing value for %s\n", a.c_str()); std::exit(2); } return argv[++i]; };
        const int i_flag = i;
        if (a == "--Z") zs = parse_z(next());
        else if (a == "--gpus") gpus = std::atoi(next());
        else if (a == "--framed") framed = true;
        else if (a == "--atom-index") atom_index = parse_z(next());
        else if (a == "--radial") radial_dir = next();
        else if (a == "--logderiv") logderiv_dir = next();
        else if (a == "--rc") rc = std::atof(next());
        else if (a == "--energies") energies = next();
        else if (a == "--pseudo") pseudo_dir = next();
        else if (a == "--pseudo-rc") pseudo_rc = next();
        else if (a == "--pseudo-test") pseudo_test = next();
        else if (a == "--pseudo-local") {
            const std::string v = next();
            if (v.size() != 1 || v[0] < '0' || v[0] > '3') { std::fprintf(stderr, "dftatom: --pseudo-local expects l = 0, 1, 2 or 3, got '%s'\n", v.c_str()); return 2; }
            pseudo_local = v[0] - '0';
        }
        else if (a == "--pseudo-core") {
            const std::string v = next();
            char* end = nullptr;
            pseudo_core = std::strtod(v.c_str(), &end);
            if (v.empty() || *end || !std::isfinite(pseudo_core) || pseudo_core < 0.) {
                std::fprintf(stderr, "dftatom: --pseudo-core expects a radius >= 0 in bohr (0 = the full core), got '%s'\n", v.c_str()); return 2;
            }
        }
        else if (a == "--charge") charge = std::atof(next());
        else if (a == "--config") config_str = next();
        else if (a == "--levels") base.levels = std::atoi(next());
        else if (a == "--delta") base.delta = std::atof(next());
        else if (a == "--mixing" || a == "--alpha") base.mixing = std::atof(next());
        else if (a == "--rmax") base.max_r = std::atof(next());
        else if (a == "--method") {         // 0 | lda, 1 | lsda; 2, 3: the same on the uniform grid (CalculateUniformLDA / LSDA, DFTAtom.h:15,18)
            std::string m = next();
            base.method = (m == "1" || m == "lsda" || m == "LSDA") ? 1 : (m == "2" ? 2 : (m == "3" ? 3 : 0));
        }
        else if (a == "--uniform") base.method |= 2;
        else if (a == "--precision") precision = std::atoi(next());
        else if (a == "--device") device = std::atoi(next());
        else if (a == "--ini") read_ini(next(), base);
        else if (a == "--json") json = true;
        else if (a == "--quiet-steps") quiet = true;
        else if (a == "--help" || a == "-h") {
            std::printf("usage: dftatom [--Z 18|1-92|a,b,c] [--levels L] [--delta d] [--mixing a] [--rmax R] [--method 0|1] "
                        "[--precision p] [--json] [--quiet-steps] [--device k] [--gpus N] [--ini file] [--radial DIR] [--charge Q] [--config \"...\"]\n"
                        "               [--logderiv DIR --rc R [--energies lo:hi:n]] [--pseudo DIR --pseudo-rc Rs[,Rp,Rd,Rf] [--pseudo-local L] [--pseudo-test \"C1;C2\"]\n"
                        "               [--pseudo-core R]]\n"
                        "  --radial DIR  write the converged r, rho, V, V_H and orbitals u(r) of every atom to DIR/<index>_Z<Z>.tsv\n"
                        "  --charge Q    solve every atom of --Z ionised by Q electrons (the reference's configuration; fractional allowed, < 0 = anion)\n"
                        "  --config C    solve one atom (a single --Z) in configuration C, e.g. \"[Ar] 3d10\", \"1s2 2s2 2p4.5\", LSDA \"[He] 2s1 2p3/1\"\n"
                        "  --logderiv DIR  write the logarithmic derivatives D_l(E) = u'(r_c)/u(r_c), l = 0..3 per spin, of every atom's converged V to\n"
                        "                DIR/<index>_Z<Z>_logderiv.tsv (columns spin l E D nodes phase u du)\n"
                        "  --rc R        radius of --logderiv in bohr (the nearest grid node is used)\n"
                        "  --energies lo:hi:n  energies of --logderiv, n points from lo to hi Hartree (default -2:1:301)\n"
                        "  --pseudo DIR  write Troullier-Martins pseudopotentials of every LDA atom (valence = largest n per l) to DIR/<index>_Z<Z>_pseudo.tsv\n"
                        "                (columns r, V_ion per l, V_scr per l, u per l, rho_val); with --logderiv also <index>_Z<Z>_pseudo_logderiv.tsv\n"
                        "  --pseudo-rc Rs[,Rp,Rd,Rf]  radii of --pseudo in bohr by l (an l beyond the list takes the last one)\n"
                        "  --pseudo-local L  Kleinman-Bylander form of --pseudo with the channel l = L local: one \"# kb\" line per channel (l E_KB cos\n"
                        "                eps_loc0 eps_loc1 ghost status) and beta columns; with --logderiv also <index>_Z<Z>_pseudo_kb_logderiv.tsv\n"
                        "  --pseudo-test \"C1;C2\"  with --pseudo and a single --Z: solve the pseudo-atom in the reference valence configuration and in\n"
                        "                each valence configuration Ck (e.g. \"3s1 3p3;3s2 3p1\"), the all-electron atom in core + each, and write\n"
                        "                <index>_Z<Z>_pseudo_test.tsv (config Q E_AE E_PS dE_AE dE_PS dE_PS-dE_AE statuses, then eps_AE / eps_PS per level)\n"
                        "  --pseudo-core R  nonlinear core correction of --pseudo: unscreen with the partial core of the other levels at R bohr (0 = the\n"
                        "                full core); --pseudo-test solves with it; adds a \"# core\" line and rho_core, rho_pc columns\n");
            return 0;
        } else { std::fprintf(stderr, "unknown flag %s\n", a.c_str()); return 2; }
        if (a != "--Z" && a != "--gpus" && a != "--device" && a != "--framed" && a != "--atom-index") for (int q = i_flag; q <= i; ++q) passthrough.push_back(argv[q]);
    }
    if (zs.empty()) zs.push_back(base.Z);
    if (!config_str.empty() && (zs.size() != 1 || charge != 0.)) { std::fprintf(stderr, "dftatom: --config needs a single --Z and no --charge\n"); return 2; }
    if (!atom_index.empty() && atom_index.size() != zs.size()) { std::fprintf(stderr, "dftatom: --atom-index needs one index per --Z entry\n"); return 2; }
    if (!radial_dir.empty() && mkdir(radial_dir.c_str(), 0777) != 0 && errno != EEXIST) { std::perror(radial_dir.c_str()); return 1; }
    std::vector<double> ld_E;
    if (!logderiv_dir.empty()) {
        double lo = 0., hi = 0.; int ne = 0; char tail = 0;
        if (std::sscanf(energies.c_str(), "%lf:%lf:%d%c", &lo, &hi, &ne, &tail) != 3 || ne < 1 || !std::isfinite(lo) || !std::isfinite(hi)) {
            std::fprintf(stderr, "dftatom: --energies expects lo:hi:n with n >= 1, got '%s'\n", energies.c_str()); return 2;
        }
        for (int k = 0; k < ne; ++k) ld_E.push_back(k == ne - 1 && ne > 1 ? hi : lo + (hi - lo) * k / (ne > 1 ? ne - 1 : 1));
        if (!(rc > 0.)) { std::fprintf(stderr, "dftatom: --logderiv needs --rc R (bohr)\n"); return 2; }
        if (mkdir(logderiv_dir.c_str(), 0777) != 0 && errno != EEXIST) { std::perror(logderiv_dir.c_str()); return 1; }
    }
    std::vector<double> ps_rc;
    if (pseudo_local >= 0 && pseudo_dir.empty()) { std::fprintf(stderr, "dftatom: --pseudo-local needs --pseudo DIR\n"); return 2; }
    if (!std::isnan(pseudo_core) && pseudo_dir.empty()) { std::fprintf(stderr, "dftatom: --pseudo-core needs --pseudo DIR\n"); return 2; }
    std::vector<std::string> ps_tests;
    if (!pseudo_test.empty()) {
        if (pseudo_dir.empty() || zs.size() != 1) { std::fprintf(stderr, "dftatom: --pseudo-test needs --pseudo DIR and a single --Z\n"); return 2; }
        if (base.method & 2) { std::fprintf(stderr, "dftatom: --pseudo-test needs the logarithmic grid (method 0)\n"); return 2; }
        for (size_t p = 0; p <= pseudo_test.size();) {
            const size_t q = std::min(pseudo_test.find(';', p), pseudo_test.size());
            const std::string t = pseudo_test.substr(p, q - p);
            dftatom_config c = {};
            if (t.find_first_not_of(" \t") == std::string::npos || !parse_config(t, 0, &c) || c.n_orbitals == 0) {
                std::fprintf(stderr, "dftatom: --pseudo-test: cannot read the configuration '%s'\n", t.c_str()); return 2;
            }
            ps_tests.push_back(t);
            p = q + 1;
        }
    }
    if (!pseudo_dir.empty()) {
        if (base.method & 1) { std::fprintf(stderr, "dftatom: --pseudo needs an LDA atom (method 0 or 2): the unscreening is spin-unpolarised\n"); return 2; }
        for (size_t p = 0; p < pseudo_rc.size();) {
            const size_t q = std::min(pseudo_rc.find(',', p), pseudo_rc.size());
            char* end = nullptr;
            const std::string tok = pseudo_rc.substr(p, q - p);
            const double x = std::strtod(tok.c_str(), &end);
            if (tok.empty() || *end || !(x > 0.)) { std::fprintf(stderr, "dftatom: --pseudo-rc expects Rs[,Rp,Rd,Rf] in bohr, got '%s'\n", pseudo_rc.c_str()); return 2; }
            ps_rc.push_back(x);
            p = q + 1;
        }
        if (ps_rc.empty() || ps_rc.size() > 4) { std::fprintf(stderr, "dftatom: --pseudo needs --pseudo-rc Rs[,Rp,Rd,Rf] (1 to 4 radii)\n"); return 2; }
        if (!logderiv_dir.empty() && rc < *std::max_element(ps_rc.begin(), ps_rc.end())) {
            std::fprintf(stderr, "dftatom: with --pseudo, --rc must be >= every --pseudo-rc radius\n"); return 2;
        }
        if (mkdir(pseudo_dir.c_str(), 0777) != 0 && errno != EEXIST) { std::perror(pseudo_dir.c_str()); return 1; }
    }
    if (gpus > 1) {
        char self[4096];
        const ssize_t len = readlink("/proc/self/exe", self, sizeof self - 1);
        if (len <= 0) { std::perror("readlink /proc/self/exe"); return 1; }
        self[len] = 0;
        return run_sharded(self, zs, base.method, gpus, passthrough, json);
    }
    const int n = (int)zs.size();
    std::vector<dftatom_options> opts(n, base);
    for (int k = 0; k < n; ++k) opts[k].Z = zs[k];
    // --charge / --config: every atom's configuration (none: the reference's Aufbau atom, dftatom_solve_batch_radial's arguments)
    const bool configured = charge != 0. || !config_str.empty();
    std::vector<dftatom_config> cfgs(configured ? n : 0);
    for (int k = 0; k < n && configured; ++k) {
        if (!config_str.empty() ? !parse_config(config_str, base.method, &cfgs[k]) : dftatom_config_aufbau(opts[k].Z, base.method, charge, &cfgs[k]) != DFTATOM_OK) {
            if (config_str.empty()) std::fprintf(stderr, "dftatom: %s\n", dftatom_last_error());
            return 2;
        }
    }

    dftatom_ctx* ctx = nullptr;
    if (dftatom_create(&ctx, device) != DFTATOM_OK) { std::fprintf(stderr, "dftatom: %s\n", dftatom_last_error()); return 1; }
    const int stride = DFTATOM_MAX_STEPS_LSDA;
    std::vector<dftatom_result> res(n);
    std::vector<dftatom_step> steps((size_t)n * stride);
    // --radial: arrays of the whole batch, rows of the orbitals in call order (dftatom_radial)
    const int N = dftatom_n_nodes(base.levels);
    std::vector<long long> row0(n + 1, 0);
    const bool export_orb = !radial_dir.empty() || !pseudo_dir.empty();
    for (int k = 0; k < n && export_orb; ++k) {
        dftatom_level la[DFTATOM_MAX_LEVELS], lb[DFTATOM_MAX_LEVELS];
        int na = 0, nb = 0, ea = 0, eb = 0;
        if (configured) na = cfgs[k].n_orbitals;
        else if (opts[k].method & 1) dftatom_split_spin(opts[k].Z, la, &na, lb, &nb, &ea, &eb);
        else na = std::max(0, dftatom_aufbau(opts[k].Z, la, DFTATOM_MAX_LEVELS));
        row0[k + 1] = row0[k] + na + nb;
    }
    std::vector<double> r_grid, rho, vks, vh, orb;
    dftatom_radial rad = {};
    if (export_orb) {
        r_grid.resize(N); rho.resize((size_t)n * 2 * N); vh.resize((size_t)n * N); orb.resize((size_t)row0[n] * N);
        rad.r = r_grid.data(); rad.rho = rho.data(); rad.v_hartree = vh.data(); rad.orbitals = orb.data(); rad.orbital_rows = row0[n];
    }
    const bool export_v = export_orb || !logderiv_dir.empty();
    if (export_v) { vks.resize((size_t)n * 2 * N); rad.v = vks.data(); }
    if (dftatom_solve_batch_config(ctx, opts.data(), configured ? cfgs.data() : nullptr, n, res.data(), steps.data(), stride,
                                   export_v ? &rad : nullptr) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: %s\n", dftatom_last_error());
        dftatom_destroy(ctx);
        return 1;
    }
    double ms = 0; long long launches = 0;
    dftatom_last_timing(ctx, &ms, &launches);
    for (int a = 0; a < n && !radial_dir.empty(); ++a)
        if (write_radial(radial_dir, atom_index.empty() ? a : atom_index[a], opts[a], res[a], N, r_grid.data(), &rho[(size_t)a * 2 * N], &vks[(size_t)a * 2 * N],
                         &vh[(size_t)a * N], &orb[(size_t)row0[a] * N])) { dftatom_destroy(ctx); return 1; }
    for (int a = 0; a < n && !logderiv_dir.empty(); ++a)
        if (write_logderiv(ctx, logderiv_dir, atom_index.empty() ? a : atom_index[a], opts[a], res[a].n_spin, &vks[(size_t)a * 2 * N], rc, ld_E)) {
            dftatom_destroy(ctx); return 1;
        }
    for (int a = 0; a < n && !pseudo_dir.empty(); ++a)
        if (write_pseudo(ctx, pseudo_dir, logderiv_dir, atom_index.empty() ? a : atom_index[a], opts[a], res[a], configured ? &cfgs[a] : nullptr, N,
                         r_grid.data(), &vks[(size_t)a * 2 * N], &orb[(size_t)row0[a] * N], ps_rc, rc, ld_E, pseudo_local, ps_tests, pseudo_core)) {
            dftatom_destroy(ctx); return 1;
        }

    if (json && !framed) std::printf("[");
    for (int a = 0; a < n; ++a) {
        const dftatom_result& R = res[a];
        if (framed) std::printf("\x1e%d\n", a);             // frame header: record separator + index into this child's atom list
        if (json) {
            std::printf("%s{\"Z\":%d,\"method\":%d,\"status\":%d,\"n_steps\":%d,\"Etotal\":%.17g,\"Ekin\":%.17g,\"Ecoul\":%.17g,\"Eenuc\":%.17g,\"Exc\":%.17g,\"levels\":[",
                        (a && !framed) ? "," : "", opts[a].Z, opts[a].method, R.status, R.n_steps, R.Etotal, R.Ekin, R.Ecoul, R.Eenuc, R.Exc);
            bool first = true;
            for (int s = 0; s < R.n_spin; ++s)
                for (int k = 0; k < R.n_levels[s]; ++k) {
                    const dftatom_level& L = R.levels[s][k];
                    if (configured)
                        std::printf("%s{\"spin\":%d,\"n\":%d,\"l\":%d,\"occ\":%.17g,\"nodes\":%d,\"E\":%.17g}", first ? "" : ",", s, L.n, L.l,
                                    exact_occ(L, s, &cfgs[a]), L.nodes, L.E);
                    else std::printf("%s{\"spin\":%d,\"n\":%d,\"l\":%d,\"occ\":%d,\"nodes\":%d,\"E\":%.17g}", first ? "" : ",", s, L.n, L.l, L.occ, L.nodes, L.E);
                    first = false;
                }
            std::printf("]");
            if (configured) {    // the atom's net charge Z - sum occ
                double q = 0.;
                for (int k = 0; k < cfgs[a].n_orbitals; ++k) q += cfgs[a].orb[k].occ;
                std::printf(",\"charge\":%.17g", opts[a].Z - q);
            }
            if (!quiet) {       // every "Step:" block of the reference's log, full precision
                std::printf(",\"steps\":[");
                for (int sp = 0; sp < R.n_steps; ++sp) {
                    const dftatom_step& S = steps[(size_t)a * stride + sp];
                    std::printf("%s{\"Etotal\":%.17g,\"Ekin\":%.17g,\"Ecoul\":%.17g,\"Eenuc\":%.17g,\"Exc\":%.17g,\"E\":[", sp ? "," : "", S.Etotal, S.Ekin, S.Ecoul,
                                S.Eenuc, S.Exc);
                    bool f1 = true;
                    for (int s2 = 0; s2 < R.n_spin; ++s2)
                        for (int k = 0; k < R.n_levels[s2]; ++k) { std::printf("%s%.17g", f1 ? "" : ",", S.E[s2][k]); f1 = false; }
                    std::printf("]}");
                }
                std::printf("]");
            }
            std::printf("}");
            continue;
        }
        const bool uni = opts[a].method >= 2, lsda = (opts[a].method & 1) != 0;
        std::printf("Computing atom with Z=%d using %s with %s grid\n", opts[a].Z, lsda ? "LSDA" : (uni ? "LDA" : "LSD"),
                    uni ? "uniform" : "non-uniform");                                                                       // DFTAtom.cpp:358,857,69,656
        for (int sp = quiet ? R.n_steps - 1 : 0; sp < R.n_steps; ++sp) {
            const dftatom_step& S = steps[(size_t)a * stride + sp];
            std::printf("Step: %d\n", sp);
            for (int s = 0; s < R.n_spin; ++s)
                for (int k = 0; k < R.n_levels[s]; ++k)
                    std::printf("Energy %s%d%c: %.*f Num nodes: %d\n", (uni && lsda) ? (s ? "beta " : "alpha ") : "", R.levels[s][k].n, kOrb[R.levels[s][k].l],
                                precision, S.E[s][k], R.levels[s][k].nodes);                                                 // tags: DFTAtom.cpp:269-277
            std::printf("Etotal = %.*f Ekin = %.*f Ecoul = %.*f Eenuc = %.*f Exc = %.*f\n", precision, S.Etotal, precision, S.Ekin, precision, S.Ecoul,
                        precision, S.Eenuc, precision, S.Exc);
            if (sp == R.n_steps - 1 && R.status == DFTATOM_CONVERGED) std::printf("\nFinished!\n\n");
            else std::printf("********************************************************************************\n");
        }
        if (opts[a].method & 1) {
            const dftatom_config* cf = configured ? &cfgs[a] : nullptr;
            std::printf("Alpha: "); print_conf(R.sorted[0], R.n_levels[0], 0, cf);
            std::printf("\nBeta: "); print_conf(R.sorted[1], R.n_levels[1], 1, cf);
        } else print_conf(R.sorted[0], R.n_levels[0], 0, configured ? &cfgs[a] : nullptr);
        std::printf("\n");
    }
    if (json && !framed) std::printf("]\n");
    std::fprintf(stderr, "dftatom: %d atom(s), device time %.2f ms, %lld kernel launches\n", n, ms, launches);
    dftatom_destroy(ctx);
    return 0;
}
