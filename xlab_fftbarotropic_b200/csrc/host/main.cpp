// main.cpp -- main.out: the reference's RK4 driver process on the xfb backend.
//
// Command line, stdout, `log` file and output file names follow /root/reference/src/main.cpp:65-328 and
// src/main-shallow-water.cpp:75-94 (the -s/-f forcing variant):
//   -I <input dir> -O <output dir> -i <initial file>      (main.cpp:68-80; -o is accepted as an alias of -O,
//                                                          README.md:36 documents lower-case flags)
//   -f <fifo> | -s <script>                                (main-shallow-water.cpp:86-93)
// Compile-time constants of src/configuration.hpp:13-36 are run-time options with the same defaults:
//   -n <NPTS=768> -d <dt=3> -t <total_steps=1200> -r <record_step=100> -L <600000> -N <NU=6.5>
// Additions: -g <cuda device>, -D (also write filamentation time / deformation factor at record steps),
//   -q (no per-step line), -c <tracer file> [-k <kappa>] (advect a passive tracer read from <input dir>, written as
//   tracer_step_N.bin after the reference's five files),
//   -b <members> (ensemble: member m starts from <initial file> with "%d" replaced by m -- or all members from the same
//      file -- and writes <field>_step_N.bin for m = 0, <field>_step_N.m<m>.bin otherwise),
//   -G <gpus> (the members are spread over that many devices starting at -g, no communication),
//   -S <ranks> (ONE grid slab-decomposed over that many GPUs: the process forks one rank per device, the ranks exchange
//      over NVLink (xfb_create_dist), each reads and writes its own rows of the field files; same files and log),
//   -E (at every record step, per member: the domain means E, Z, P appended to <output>/integrals.txt as
//      `step time member E Z P`, and the isotropic shell spectra written to <output>/spectrum_step_N.txt -- .m<m>.txt for
//      members other than 0 -- one `s k[1/m] E(s) Z(s)` line per shell; neither goes into `log`.  A non-finite total
//      stops the run with exit status 1 once the record files already issued are written).
//   -T (at every record step, per member: the spectral budget of xfb_get_spectral_budget -- the rates of E and Z from the
//      nonlinear transfer T, the forcing F (the source the handle holds) and the dissipation D -- written to
//      <output>/budget_step_N.txt (.m<m>.txt for members other than 0), one `s k[1/m] T_E F_E D_E T_Z F_Z D_Z Pi_E Pi_Z`
//      line per shell with the fluxes Pi(s) = -sum_{s' <= s} T(s'), and the domain totals appended to <output>/budget.txt
//      as `step time member T_E F_E D_E T_Z F_Z D_Z`; neither goes into `log`).
//   -B <beta> -R <mu> -H <nu_h> -P <order=4> (linear terms of the vorticity equation, xfb_set_linear_terms: beta-plane
//      [1/(m s)], linear drag [1/s], hyperviscosity nu_h (-lap)^order [m^(2 order)/s], order 1..8; on every handle of the
//      run, -b, -G and -S ranks included.  An invalid value stops with exit status 1 before any step.  Without these
//      flags the run is the reference's equation and its output is unchanged).
// Record output is asynchronous (SURVEY.md 8f-2): at a record step the five fields are formed on the GPU and copied
// to pinned host buffers on a second stream (xfb_get_field_async) while the next stretch of steps already runs; a
// writer thread waits for each buffer, calls writeField and appends the `log` line -- same files, same order as the
// reference (main.cpp:266-282,183-222).
// All arithmetic runs on the GPU through the C ABI (include/xfb.h); this file is I/O and control only.
#include <fcntl.h>
#include <getopt.h>
#include <sys/wait.h>
#include <unistd.h>

#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/xfb.h"
#include "fieldio.hpp"
#include "vorticity_source.hpp"

using namespace VORT_SRC_READER;

#define CHECK(call)                                                        \
    do {                                                                   \
        if ((call) != 0) {                                                 \
            std::fprintf(stderr, "main.out: %s\n", xfb_last_error());      \
            return 1;                                                      \
        }                                                                  \
    } while (0)

// -E: number of shells that holds every mode of an n x n grid (the shell of (n/2, n/2) plus one, integer rule)
static int all_shells(int n)
{
    const long long m = 2LL * (n / 2) * (n / 2);
    long long s = (long long)std::sqrt((double)m);
    while (s * s > m) --s;
    while ((s + 1) * (s + 1) <= m) ++s;
    return (int)(s + (m > s * s + s ? 1 : 0) + 1);
}

// -E at one record step for one member: spectrum file, integrals line; returns 1 if a total is not finite
static int write_energy(const std::string &output, FILE *integrals, int step, float dt, int member, float L, const double *tot,
                        const std::vector<double> &e, const std::vector<double> &z)
{
    char name[1024];
    if (member == 0) std::snprintf(name, sizeof(name), "%s/spectrum_step_%d.txt", output.c_str(), step);
    else std::snprintf(name, sizeof(name), "%s/spectrum_step_%d.m%d.txt", output.c_str(), step, member);
    if (FILE *f = std::fopen(name, "w")) {
        std::fprintf(f, "# s  k[1/m]  E(s)  Z(s)   (step %d, member %d; shell sums of E = <u^2+v^2>/2 and Z = <zeta^2>/2)\n", step, member);
        const double dk = 2.0 * M_PI / (double)L;
        for (size_t k = 0; k < e.size(); ++k) std::fprintf(f, "%zu %.9g %.17g %.17g\n", k, dk * (double)k, e[k], z[k]);
        std::fclose(f);
    }
    if (integrals) {
        std::fprintf(integrals, "%d %.17g %d %.17g %.17g %.17g\n", step, (double)step * dt, member, tot[0], tot[1], tot[2]);
        std::fflush(integrals);
    }
    return (std::isfinite(tot[0]) && std::isfinite(tot[1]) && std::isfinite(tot[2])) ? 0 : 1;
}

// -T at one record step for one member: budget file with the fluxes formed here, totals line
static void write_budget(const std::string &output, FILE *totals_file, int step, float dt, int member, float L, const double *tot,
                         const std::vector<double> &b)
{
    const size_t nsh = b.size() / XFB_BUDGET_N;
    char name[1024];
    if (member == 0) std::snprintf(name, sizeof(name), "%s/budget_step_%d.txt", output.c_str(), step);
    else std::snprintf(name, sizeof(name), "%s/budget_step_%d.m%d.txt", output.c_str(), step, member);
    if (FILE *f = std::fopen(name, "w")) {
        std::fprintf(f, "# s  k[1/m]  T_E  F_E  D_E  T_Z  F_Z  D_Z  Pi_E  Pi_Z   (step %d, member %d; shell sums of the rates of "
                        "E and Z, Pi(s) = -sum of T up to s)\n", step, member);
        const double dk = 2.0 * M_PI / (double)L;
        double pe = 0.0, pz = 0.0;
        for (size_t k = 0; k < nsh; ++k) {
            pe -= b[XFB_BUDGET_TE * nsh + k];
            pz -= b[XFB_BUDGET_TZ * nsh + k];
            std::fprintf(f, "%zu %.9g", k, dk * (double)k);
            for (int q = 0; q < XFB_BUDGET_N; ++q) std::fprintf(f, " %.17g", b[q * nsh + k]);
            std::fprintf(f, " %.17g %.17g\n", pe, pz);
        }
        std::fclose(f);
    }
    if (totals_file) {
        std::fprintf(totals_file, "%d %.17g %d", step, (double)step * dt, member);
        for (int q = 0; q < XFB_BUDGET_N; ++q) std::fprintf(totals_file, " %.17g", tot[q]);
        std::fprintf(totals_file, "\n");
        std::fflush(totals_file);
    }
}

// -B -R -H -P: the linear terms, applied to every handle the run creates
struct LinOpts {
    bool set;
    float beta, mu, nu_h;
    int order;
};

static int set_linear(xfb_handle h, const LinOpts &lin)
{
    return lin.set ? xfb_set_linear_terms(h, lin.beta, lin.mu, lin.nu_h, lin.order) : 0;
}

// a finite float option value; false on trailing characters or an unparsable / non-finite value
static bool parse_float(const char *s, float *out)
{
    char *end = nullptr;
    const double v = std::strtod(s, &end);
    if (end == s || *end != '\0' || !std::isfinite(v) || !std::isfinite((float)v)) return false;
    *out = (float)v;
    return true;
}

struct SlabOpts {
    std::string input, output, init_file;
    int npts, record_step, total_steps, device, ranks;
    float L, NU, dt;
    bool diagnostics, quiet, energy, budget;
    LinOpts lin;
};

// one rank of `-S <ranks>`: local rows [row0, row0 + rows) of every file
static int slab_rank(const SlabOpts &o, int rank, const char *id128)
{
    const int n = o.npts;
    int row0 = 0, rows = 0, nchunks = 8;
    while (nchunks > 1 && ((n / o.ranks) % nchunks != 0 || ((n / o.ranks) / nchunks) % 2 != 0)) nchunks /= 2;
    xfb_handle h = nullptr;
    CHECK(xfb_create_dist(&h, n, n, o.L, o.L, o.NU, o.device + rank, rank, o.ranks, nchunks, id128));
    CHECK(set_linear(h, o.lin));                                   // per rank, the same values everywhere
    CHECK(xfb_slab_partition(n, n, o.ranks, nchunks, rank, &row0, &rows, nullptr, nullptr, nullptr, nullptr));
    const size_t local = (size_t)rows * n;
    const off_t off = (off_t)row0 * n * (off_t)sizeof(float);
    std::vector<float> buf(local);
    char filename[1024];
    std::snprintf(filename, sizeof(filename), "%s/%s", o.input.c_str(), o.init_file.c_str());
    {
        const int fd = open(filename, O_RDONLY);
        if (fd < 0 || pread(fd, buf.data(), local * sizeof(float), off) != (ssize_t)(local * sizeof(float))) {
            std::fprintf(stderr, "main.out: rank %d cannot read its rows of %s\n", rank, filename);
            return 1;
        }
        close(fd);
    }
    FILE *log_fd = rank == 0 ? std::fopen("log", "w") : nullptr;
    FILE *integrals = nullptr;
    if (o.energy && rank == 0) {
        std::snprintf(filename, sizeof(filename), "%s/integrals.txt", o.output.c_str());
        integrals = std::fopen(filename, "w");
    }
    const int nsh = o.energy ? all_shells(n) : 0;
    std::vector<double> es(nsh), zs(nsh);
    FILE *budget_file = nullptr;
    if (o.budget && rank == 0) {
        std::snprintf(filename, sizeof(filename), "%s/budget.txt", o.output.c_str());
        budget_file = std::fopen(filename, "w");
    }
    std::vector<double> bs(o.budget ? (size_t)XFB_BUDGET_N * all_shells(n) : 0);
    CHECK(xfb_set_vorticity(h, 0, buf.data()));
    if (rank == 0) std::printf("Initialization complete.\n");
    auto record = [&](const char *stem, int which, int step) -> int {
        if (xfb_get_field(h, 0, which, buf.data()) != 0) return 1;            // collective: local rows
        std::snprintf(filename, sizeof(filename), "%s/%s_step_%d.bin", o.output.c_str(), stem, step);
        const int fd = open(filename, O_WRONLY | O_CREAT, 0644);
        if (fd < 0 || pwrite(fd, buf.data(), local * sizeof(float), off) != (ssize_t)(local * sizeof(float))) {
            std::fprintf(stderr, "main.out: rank %d cannot write its rows of %s\n", rank, filename);
            return 1;
        }
        close(fd);
        if (log_fd) { std::fprintf(log_fd, "%s\n", filename); std::fflush(log_fd); }
        return 0;
    };
    for (int step = 0; step < o.total_steps;) {
        const bool record_flag = (step % o.record_step) == 0;
        if (rank == 0 && !o.quiet) std::printf("# Step %d, time = %.2f%s\n", step, step * o.dt, record_flag ? ", record now!" : "");
        if (record_flag) {
            if (record("vort_src_input", XFB_SRC, step) || record("vort", XFB_VORT, step) || record("psi", XFB_PSI, step) ||
                record("u", XFB_U, step) || record("v", XFB_V, step) ||
                (o.diagnostics && (record("tfil", XFB_TFIL, step) || record("deform", XFB_DEFORM, step)))) {
                std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                return 1;
            }
            if (o.energy) {
                double tot[3];
                CHECK(xfb_get_energy_spectrum(h, 0, XFB_VORT, nsh, tot, es.data(), zs.data()));      // collective
                const bool bad = !(std::isfinite(tot[0]) && std::isfinite(tot[1]) && std::isfinite(tot[2]));
                if (rank == 0) write_energy(o.output, integrals, step, o.dt, 0, o.L, tot, es, zs);
                if (bad) {
                    if (rank == 0) std::fprintf(stderr, "main.out: non-finite energy/enstrophy at step %d (member 0)\n", step);
                    if (integrals) std::fclose(integrals);
                    if (log_fd) std::fclose(log_fd);
                    xfb_sync(h);
                    xfb_destroy(h);
                    return 1;
                }
            }
            if (o.budget) {
                double tot[XFB_BUDGET_N];
                CHECK(xfb_get_spectral_budget(h, 0, (int)(bs.size() / XFB_BUDGET_N), tot, bs.data()));      // collective
                if (rank == 0) write_budget(o.output, budget_file, step, o.dt, 0, o.L, tot, bs);
            }
        }
        const int next_record = (step / o.record_step + 1) * o.record_step;
        const int chunk = (next_record < o.total_steps ? next_record : o.total_steps) - step;
        if (rank == 0 && !o.quiet)
            for (int s = step + 1; s < step + chunk; ++s) std::printf("# Step %d, time = %.2f\n", s, s * o.dt);
        CHECK(xfb_step(h, chunk, o.dt));
        step += chunk;
    }
    CHECK(xfb_sync(h));
    if (log_fd) std::fclose(log_fd);
    if (integrals) std::fclose(integrals);
    if (budget_file) std::fclose(budget_file);
    xfb_destroy(h);
    if (rank == 0) std::printf("Program ends. Congrats!\n");
    return 0;
}

// -S <ranks>: fork one process per GPU BEFORE any CUDA call; rank 0 hands the NCCL unique id to the others through pipes
static int run_slab(const SlabOpts &o)
{
    if (o.ranks > 16 || o.npts % (2 * o.ranks) != 0) {
        std::fprintf(stderr, "main.out: -S %d does not divide a %d^2 grid into whole row pairs\n", o.ranks, o.npts);
        return 1;
    }
    std::fflush(stdout);
    int pipes[16][2];
    for (int r = 1; r < o.ranks; ++r)
        if (pipe(pipes[r]) != 0) { perror("pipe"); return 1; }
    std::vector<pid_t> kids;
    for (int r = 0; r < o.ranks; ++r) {
        const pid_t pid = fork();
        if (pid < 0) { perror("fork"); return 1; }
        if (pid == 0) {
            char id[128];
            if (r == 0) {
                if (xfb_nccl_unique_id(id) != 0) { std::fprintf(stderr, "main.out: %s\n", xfb_last_error()); _exit(1); }
                for (int q = 1; q < o.ranks; ++q)
                    if (write(pipes[q][1], id, 128) != 128) _exit(1);
            } else if (read(pipes[r][0], id, 128) != 128) _exit(1);
            const int rc = slab_rank(o, r, id);
            std::fflush(stdout);
            _exit(rc);
        }
        kids.push_back(pid);
    }
    int worst = 0;
    for (pid_t k : kids) {
        int st = 0;
        waitpid(k, &st, 0);
        if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) worst = 1;
    }
    return worst;
}

int main(int argc, char *args[])
{
    std::string input = "input", output = "output", init_file = "initial_vorticity.bin";   // configuration.hpp:39-41
    std::string vort_src_filename, tracer_file;
    float kappa = -1.0f;
    RECIPE_TYPE recipe_type = EMPTY;
    int npts = 768, record_step = 100, total_steps = -1, device = 0, members = 1, ngpus = 1, slab_ranks = 0;
    float L = 600000.0f, NU = 6.5f, dt = 3.0f;
    bool diagnostics = false, quiet = false, energy = false, budget = false;
    LinOpts lin{false, 0.0f, 0.0f, 0.0f, 4};
    bool bad_lin = false;

    int opt;
    while ((opt = getopt(argc, args, "I:O:o:i:s:f:n:d:t:r:L:N:g:c:k:b:G:S:B:R:H:P:DETq")) != EOF) {
        switch (opt) {
        case 'I': input = optarg; break;
        case 'O': case 'o': output = optarg; break;
        case 'i': init_file = optarg; break;
        case 's': vort_src_filename = optarg; recipe_type = SCRIPT; break;
        case 'f': vort_src_filename = optarg; recipe_type = FIFO; break;
        case 'n': npts = std::atoi(optarg); break;
        case 'd': dt = (float)std::atof(optarg); break;
        case 't': total_steps = std::atoi(optarg); break;
        case 'r': record_step = std::atoi(optarg); break;
        case 'L': L = (float)std::atof(optarg); break;
        case 'N': NU = (float)std::atof(optarg); break;
        case 'g': device = std::atoi(optarg); break;
        case 'c': tracer_file = optarg; break;        // passive tracer: initial field <input>/<file>, tracer_step_N.bin
        case 'k': kappa = (float)std::atof(optarg); break;   // its diffusivity (default: NU)
        case 'b': members = std::atoi(optarg); break;
        case 'G': ngpus = std::atoi(optarg); break;
        case 'S': slab_ranks = std::atoi(optarg); break;
        case 'D': diagnostics = true; break;
        case 'E': energy = true; break;
        case 'T': budget = true; break;
        case 'q': quiet = true; break;
        case 'B': lin.set = true; bad_lin |= !parse_float(optarg, &lin.beta); break;
        case 'R': lin.set = true; bad_lin |= !parse_float(optarg, &lin.mu) || lin.mu < 0.0f; break;
        case 'H': lin.set = true; bad_lin |= !parse_float(optarg, &lin.nu_h) || lin.nu_h < 0.0f; break;
        case 'P': {
            lin.set = true;
            char *end = nullptr;
            const long v = std::strtol(optarg, &end, 10);
            if (end == optarg || *end != '\0' || v < 1 || v > 8) bad_lin = true;
            else lin.order = (int)v;
            break;
        }
        }
    }
    if (bad_lin) {
        std::fprintf(stderr, "main.out: -B <beta> -R <mu> -H <nu_h> -P <order>: finite numbers, mu >= 0, nu_h >= 0, order 1..8\n");
        return 1;
    }
    if (total_steps < 0) total_steps = (int)(60 * 60 / dt);          // configuration.hpp:36
    if (record_step < 1) record_step = 1;
    if (members < 1) members = 1;
    if (ngpus < 1) ngpus = 1;
    if (ngpus > members) ngpus = members;
    const size_t GRIDS = (size_t)npts * npts;
    const float dx = L / npts, dy = L / npts;

    std::printf("##### Model setting #####\n");
    std::printf("Initial file          : %s \n", init_file.c_str());
    std::printf("Input folder          : %s \n", input.c_str());
    std::printf("Output folder         : %s \n", output.c_str());
    std::printf("Length X              : %.3f [m]\n", L);
    std::printf("Length Y              : %.3f [m]\n", L);
    std::printf("Spatial Resolution dx : %.3f [m]\n", dx);      // the reference prints 0 here (main.cpp:89-90 before :140)
    std::printf("Spatial Resolution dy : %.3f [m]\n", dy);
    std::printf("Time Resolution dt    : %.3f [s]\n", dt);
    std::printf("#########################\n\n\n");
    std::printf("Start project.\n");

    if (slab_ranks > 1) {
        if (recipe_type != EMPTY || !tracer_file.empty() || members > 1) {
            std::fprintf(stderr, "main.out: -S (slab decomposition) runs one member without forcing or tracer\n");
            return 1;
        }
        SlabOpts so{input, output, init_file, npts, record_step, total_steps, device, slab_ranks, L, NU, dt, diagnostics, quiet,
                    energy, budget, lin};
        return run_slab(so);
    }

    FILE *log_fd = std::fopen("log", "w");                        // main.cpp:97, in the CWD
    if (log_fd == NULL) perror("Open log file");
    FILE *integrals = nullptr;                                      // -E
    if (energy) {
        const std::string name = output + "/integrals.txt";
        integrals = std::fopen(name.c_str(), "w");
        if (!integrals) perror("Open integrals.txt");
    }
    const int nsh = energy ? all_shells(npts) : 0;
    std::vector<double> es(nsh), zs(nsh);
    FILE *budget_file = nullptr;                                    // -T
    if (budget) {
        const std::string name = output + "/budget.txt";
        budget_file = std::fopen(name.c_str(), "w");
        if (!budget_file) perror("Open budget.txt");
    }
    std::vector<double> bs(budget ? (size_t)XFB_BUDGET_N * all_shells(npts) : 0);

    // ensemble members in blocks over the devices: handle d holds members [first[d], first[d] + count[d])
    std::vector<xfb_handle> hs(ngpus, nullptr);
    std::vector<int> first(ngpus), count(ngpus);
    for (int d = 0; d < ngpus; ++d) {
        first[d] = (int)((long long)members * d / ngpus);
        count[d] = (int)((long long)members * (d + 1) / ngpus) - first[d];
        CHECK(xfb_create(&hs[d], npts, npts, L, L, NU, count[d], device + d));
        CHECK(set_linear(hs[d], lin));
    }
    auto owner = [&](int m, int *local) { int d = 0; while (m >= first[d] + count[d]) ++d; *local = m - first[d]; return hs[d]; };
    xfb_handle h = hs[0];

    std::vector<float> field(GRIDS);
    // the forcing field of a step is read from the recipe stream straight into page-locked memory: its upload then runs at
    // the full PCIe rate (a pageable 8192^2 field takes several step times)
    float *src = nullptr;
    if (recipe_type != EMPTY) {
        CHECK(xfb_host_alloc(&src, GRIDS));
        std::memset(src, 0, sizeof(float) * GRIDS);
    }
    char filename[1024], pattern[1024];
    VortSrcRecipeReader vs_reader;
    if (vs_reader.init(recipe_type, vort_src_filename, GRIDS) != 0) return 1;
    for (int m = 0; m < members; ++m) {
        std::snprintf(pattern, sizeof(pattern), "%s/%s", input.c_str(), init_file.c_str());
        if (std::strstr(pattern, "%d")) std::snprintf(filename, sizeof(filename), pattern, m);      // per-member initial files
        else std::snprintf(filename, sizeof(filename), "%s", pattern);
        if (m == 0 || std::strstr(pattern, "%d")) {
            if (readFieldChecked(filename, field.data(), GRIDS) != 0) {
                std::fprintf(stderr, "main.out: cannot read the initial field %s\n", filename);
                return 1;
            }
        }
        int lm = 0;
        xfb_handle hm = owner(m, &lm);
        CHECK(xfb_set_vorticity(hm, lm, field.data()));             // step 01, main.cpp:256
    }
    std::printf("Initialization complete.\n");

    const bool tracer = !tracer_file.empty();
    if (tracer) {
        std::snprintf(filename, sizeof(filename), "%s/%s", input.c_str(), tracer_file.c_str());
        if (readFieldChecked(filename, field.data(), GRIDS) != 0) {
            std::fprintf(stderr, "main.out: cannot read the tracer field %s\n", filename);
            return 1;
        }
        for (int m = 0; m < members; ++m) {
            int lm = 0;
            xfb_handle hm = owner(m, &lm);
            CHECK(xfb_set_tracer(hm, lm, field.data(), kappa >= 0.0f ? kappa : NU));
        }
    }

    // ---- asynchronous record output: one pinned buffer per field kind, a writer thread, jobs in log order
    struct Job { xfb_handle h; int ticket; float *buf; std::string file; };
    std::deque<Job> jobs;
    std::mutex mu;
    std::condition_variable cv_jobs, cv_idle;
    bool closing = false, writer_failed = false;
    std::string writer_error;          // xfb_last_error() is thread-local: the writer thread keeps its own copy
    int pending = 0;
    std::thread writer([&]() {
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_jobs.wait(lk, [&] { return closing || !jobs.empty(); });
                if (jobs.empty()) return;
                j = jobs.front();
                jobs.pop_front();
            }
            if (xfb_wait_field(j.h, j.ticket) != 0) {
                std::lock_guard<std::mutex> lk(mu);
                if (!writer_failed) writer_error = xfb_last_error();
                writer_failed = true;
            }
            writeField(j.file.c_str(), j.buf, GRIDS);
            if (log_fd) { std::fprintf(log_fd, "%s\n", j.file.c_str()); std::fflush(log_fd); }
            {
                std::lock_guard<std::mutex> lk(mu);
                --pending;
            }
            cv_idle.notify_all();
        }
    });
    auto wait_writer = [&]() {
        std::unique_lock<std::mutex> lk(mu);
        cv_idle.wait(lk, [&] { return pending == 0; });
    };
    const int NKIND = 8;
    std::vector<float *> pinned((size_t)NKIND * members, nullptr);       // one buffer per (field kind, member)
    auto record = [&](int kind, const char *stem, int which, int step) -> int {
        for (int m = 0; m < members; ++m) {
            float *&pb = pinned[(size_t)kind * members + m];
            if (!pb && xfb_host_alloc(&pb, GRIDS) != 0) return 1;
            int ticket = -1, lm = 0;
            xfb_handle hm = owner(m, &lm);
            if (xfb_get_field_async(hm, lm, which, pb, &ticket) != 0) return 1;
            if (m == 0) std::snprintf(filename, sizeof(filename), "%s/%s_step_%d.bin", output.c_str(), stem, step);
            else std::snprintf(filename, sizeof(filename), "%s/%s_step_%d.m%d.bin", output.c_str(), stem, step, m);
            {
                std::lock_guard<std::mutex> lk(mu);
                jobs.push_back(Job{hm, ticket, pb, filename});
                ++pending;
            }
            cv_jobs.notify_one();
        }
        return 0;
    };
    auto shutdown_writer = [&]() {
        {
            std::lock_guard<std::mutex> lk(mu);
            closing = true;
        }
        cv_jobs.notify_all();
        writer.join();
    };

    int step = 0;
    while (step < total_steps) {
        const bool record_flag = (step % record_step) == 0;
        if (!quiet) {
            std::printf("# Step %d, time = %.2f", step, step * dt);
            if (record_flag) std::printf(", record now!");
            std::printf("\n");
        }
        if (record_flag) {
            wait_writer();                     // the pinned buffers of the previous record step are on disk
            // same order as the reference's log: source, vort (main.cpp:268-278), then psi, u, v (:183-222)
            if (record(0, "vort_src_input", XFB_SRC, step) || record(1, "vort", XFB_VORT, step) ||
                record(2, "psi", XFB_PSI, step) || record(3, "u", XFB_U, step) || record(4, "v", XFB_V, step) ||
                (diagnostics && (record(5, "tfil", XFB_TFIL, step) || record(6, "deform", XFB_DEFORM, step))) ||
                (tracer && record(7, "tracer", XFB_TRACER, step))) {
                std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                shutdown_writer();
                return 1;
            }
            for (int m = 0; energy && m < members; ++m) {
                int lm = 0;
                xfb_handle hm = owner(m, &lm);
                double tot[3];
                if (xfb_get_energy_spectrum(hm, lm, XFB_VORT, nsh, tot, es.data(), zs.data()) != 0) {
                    std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                    shutdown_writer();
                    return 1;
                }
                if (write_energy(output, integrals, step, dt, m, L, tot, es, zs)) {
                    std::fprintf(stderr, "main.out: non-finite energy/enstrophy at step %d (member %d)\n", step, m);
                    wait_writer();                 // the record files already issued reach the disk
                    shutdown_writer();
                    if (integrals) std::fclose(integrals);
                    if (log_fd) std::fclose(log_fd);
                    return 1;
                }
            }
            for (int m = 0; budget && m < members; ++m) {
                int lm = 0;
                xfb_handle hm = owner(m, &lm);
                double tot[XFB_BUDGET_N];
                if (xfb_get_spectral_budget(hm, lm, (int)(bs.size() / XFB_BUDGET_N), tot, bs.data()) != 0) {
                    std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                    shutdown_writer();
                    return 1;
                }
                write_budget(output, budget_file, step, dt, m, L, tot, bs);
            }
        }
        int chunk = 1;
        if (recipe_type == EMPTY) {
            // no per-step host work until the next record step: run the whole stretch on the device
            const int next_record = (step / record_step + 1) * record_step;
            chunk = (next_record < total_steps ? next_record : total_steps) - step;
            if (!quiet)
                for (int s = step + 1; s < step + chunk; ++s) std::printf("# Step %d, time = %.2f\n", s, s * dt);
        } else {
            const int got = vs_reader.read(step * dt, src);       // main-shallow-water.cpp:304
            if (got < 0) {
                // a short read of the forcing stream: the reference ignores the return value and integrates on with a
                // half-filled buffer (vorticity_source.cpp:116-126); stopping is the safe reading of that
                std::fprintf(stderr, "main.out: forcing stream ended inside a field at step %d\n", step);
                shutdown_writer();
                return 1;
            }
            for (int m = 0; got == 1 && m < members; ++m) {            // the same forcing for every member
                int lm = 0;
                xfb_handle hm = owner(m, &lm);
                if (xfb_set_source(hm, lm, src) != 0) {
                    std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                    shutdown_writer();
                    return 1;
                }
            }
        }
        for (xfb_handle hd : hs)                                       // asynchronous: the devices step concurrently
            if (xfb_step(hd, chunk, dt) != 0) {
                std::fprintf(stderr, "main.out: %s\n", xfb_last_error());
                shutdown_writer();
                return 1;
            }
        step += chunk;
    }
    int sync_rc = 0;
    for (xfb_handle hd : hs) sync_rc |= xfb_sync(hd);
    wait_writer();
    shutdown_writer();
    if (sync_rc != 0 || writer_failed) {
        std::fprintf(stderr, "main.out: %s\n", writer_failed ? writer_error.c_str() : xfb_last_error());
        return 1;
    }
    for (float *pb : pinned) xfb_host_free(pb);
    xfb_host_free(src);
    if (log_fd) std::fclose(log_fd);
    if (integrals) std::fclose(integrals);
    if (budget_file) std::fclose(budget_file);
    for (xfb_handle hd : hs) xfb_destroy(hd);
    (void)h;
    std::printf("Program ends. Congrats!\n");
    return 0;
}
