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
#include <algorithm>
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

static void print_conf(const dftatom_level* lv, int n)
{
    for (int k = 0; k < n; ++k) std::printf("%d%c%d ", lv[k].n, kOrb[lv[k].l], lv[k].occ);
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

int main(int argc, char** argv)
{
    dftatom_options base = { 36, 12, 10.0, 0.001, 0.5, 0 };     // Options.cpp:6
    std::vector<int> zs, atom_index;                        // atom_index: positions of this shard's atoms in the parent's --Z list (--gpus children)
    std::string radial_dir;
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
                        "[--precision p] [--json] [--quiet-steps] [--device k] [--gpus N] [--ini file] [--radial DIR]\n"
                        "  --radial DIR  write the converged r, rho, V, V_H and orbitals u(r) of every atom to DIR/<index>_Z<Z>.tsv\n");
            return 0;
        } else { std::fprintf(stderr, "unknown flag %s\n", a.c_str()); return 2; }
        if (a != "--Z" && a != "--gpus" && a != "--device" && a != "--framed" && a != "--atom-index") for (int q = i_flag; q <= i; ++q) passthrough.push_back(argv[q]);
    }
    if (zs.empty()) zs.push_back(base.Z);
    if (!atom_index.empty() && atom_index.size() != zs.size()) { std::fprintf(stderr, "dftatom: --atom-index needs one index per --Z entry\n"); return 2; }
    if (!radial_dir.empty() && mkdir(radial_dir.c_str(), 0777) != 0 && errno != EEXIST) { std::perror(radial_dir.c_str()); return 1; }
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

    dftatom_ctx* ctx = nullptr;
    if (dftatom_create(&ctx, device) != DFTATOM_OK) { std::fprintf(stderr, "dftatom: %s\n", dftatom_last_error()); return 1; }
    const int stride = DFTATOM_MAX_STEPS_LSDA;
    std::vector<dftatom_result> res(n);
    std::vector<dftatom_step> steps((size_t)n * stride);
    // --radial: arrays of the whole batch, rows of the orbitals in call order (dftatom_radial)
    const int N = dftatom_n_nodes(base.levels);
    std::vector<long long> row0(n + 1, 0);
    for (int k = 0; k < n && !radial_dir.empty(); ++k) {
        dftatom_level la[DFTATOM_MAX_LEVELS], lb[DFTATOM_MAX_LEVELS];
        int na = 0, nb = 0, ea = 0, eb = 0;
        if (opts[k].method & 1) dftatom_split_spin(opts[k].Z, la, &na, lb, &nb, &ea, &eb);
        else na = std::max(0, dftatom_aufbau(opts[k].Z, la, DFTATOM_MAX_LEVELS));
        row0[k + 1] = row0[k] + na + nb;
    }
    std::vector<double> r_grid, rho, vks, vh, orb;
    dftatom_radial rad = {};
    if (!radial_dir.empty()) {
        r_grid.resize(N); rho.resize((size_t)n * 2 * N); vks.resize((size_t)n * 2 * N); vh.resize((size_t)n * N); orb.resize((size_t)row0[n] * N);
        rad.r = r_grid.data(); rad.rho = rho.data(); rad.v = vks.data(); rad.v_hartree = vh.data(); rad.orbitals = orb.data(); rad.orbital_rows = row0[n];
    }
    if (dftatom_solve_batch_radial(ctx, opts.data(), n, res.data(), steps.data(), stride, radial_dir.empty() ? nullptr : &rad) != DFTATOM_OK) {
        std::fprintf(stderr, "dftatom: %s\n", dftatom_last_error());
        dftatom_destroy(ctx);
        return 1;
    }
    double ms = 0; long long launches = 0;
    dftatom_last_timing(ctx, &ms, &launches);
    for (int a = 0; a < n && !radial_dir.empty(); ++a)
        if (write_radial(radial_dir, atom_index.empty() ? a : atom_index[a], opts[a], res[a], N, r_grid.data(), &rho[(size_t)a * 2 * N], &vks[(size_t)a * 2 * N],
                         &vh[(size_t)a * N], &orb[(size_t)row0[a] * N])) { dftatom_destroy(ctx); return 1; }

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
                    std::printf("%s{\"spin\":%d,\"n\":%d,\"l\":%d,\"occ\":%d,\"nodes\":%d,\"E\":%.17g}", first ? "" : ",", s, L.n, L.l, L.occ, L.nodes, L.E);
                    first = false;
                }
            std::printf("]");
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
            std::printf("Alpha: "); print_conf(R.sorted[0], R.n_levels[0]);
            std::printf("\nBeta: "); print_conf(R.sorted[1], R.n_levels[1]);
        } else print_conf(R.sorted[0], R.n_levels[0]);
        std::printf("\n");
    }
    if (json && !framed) std::printf("]\n");
    std::fprintf(stderr, "dftatom: %d atom(s), device time %.2f ms, %lld kernel launches\n", n, ms, launches);
    dftatom_destroy(ctx);
    return 0;
}
