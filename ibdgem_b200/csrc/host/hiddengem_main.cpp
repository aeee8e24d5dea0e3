// hiddengem — command-line front-end for the batched three-state Viterbi of the engine.  Same
// options, defaults, messages and stdout table as the reference (src/hiddengem.c:13-25, 171-288).
// The recursion runs on the GPU in log space (hiddengem_viterbi_batch); the reference's x87
// long-double running products are re-synthesised for printing from their logarithms.
// Additive: -s may be given several times; the tables are read in parallel, scored in one batch and
// printed in order (formatted in parallel).  --posterior (additive) also prints each bin's posterior state
// probabilities (hiddengem_posterior_batch) and the expected state fractions.  --tracts FILE (additive) writes the IBD
// tracts, maximal runs of one state, to FILE (hiddengem_tracts_batch); stdout is unchanged.  --share-sd (additive,
// with --posterior) runs hiddengem_posterior_moments_batch in place of hiddengem_posterior_batch and adds the
// standard deviations of the posterior state shares and of the kinship, per table and over all tables.
// --tract-counts (additive, with --posterior) also runs hiddengem_tract_counts_batch and adds the posterior expected
// number of IBD tracts per state with its sd and the expected switches between states, per table and over all tables.
// --tract-lengths X1,X2,... (additive, with --posterior) also runs hiddengem_tract_lengths_batch on the START / END
// columns and adds the posterior expected number of IBD tracts at least X bp long per state, per table and over all
// tables.
#include <getopt.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/ibdgem_b200.h"
#include "textio.h"

using namespace ibdhost;

namespace {

void print_help(int code) {
    fputs("HIDDENGEM: Finds most probable path of IBD states across genomic segments.\n\n"
          "Usage: ./hiddengem -s [summary-file] [other options...] >[out-file]\n"
          "--summary, -s  FILE      Summary file from IBDGem likelihood calculation (*.summary.txt) (required)\n"
          "--p01  FLOAT             Penalty for switching between states IBD0 and IBD1 (default: 1e-3)\n"
          "--p02  FLOAT             Penalty for switching between states IBD0 and IBD2 (default: 1e-6)\n"
          "--p12  FLOAT             Penalty for switching between states IBD1 and IBD2 (default: 1e-3)\n"
          "--posterior              Also print each segment's posterior probability of every state (columns\n"
          "                            P_IBD0, P_IBD1, P_IBD2) and the expected share of segments per state\n"
          "--share-sd               With --posterior: also print the standard deviation of each state's share\n"
          "                            of segments and the window-share kinship (N_IBD1/4 + N_IBD2/2)/n with its\n"
          "                            standard deviation, from the posterior covariance; with several -s, also\n"
          "                            these figures over all tables together\n"
          "--tract-counts           With --posterior: also print the posterior expected number of IBD tracts\n"
          "                            (maximal runs of segments in one state) per state with its standard\n"
          "                            deviation, and the expected number of switches between each two states;\n"
          "                            with several -s, also these figures over all tables together\n"
          "--tract-lengths  X1,X2,...\n"
          "                         With --posterior: also print the posterior expected number of IBD tracts per\n"
          "                            state at least X bp long (END of the last segment - START of the first + 1),\n"
          "                            for up to 16 strictly increasing positive integers X; with several -s, also\n"
          "                            these figures over all tables together\n"
          "--tracts  FILE           Also write the IBD tracts (maximal runs of segments in one state) to FILE: per\n"
          "                            tract its summary file, state, first and last segment, START, END, number\n"
          "                            of segments and sites, LOD10 of its state against the next best (and with\n"
          "                            --posterior the mean and minimum posterior of its state)\n"
          "--help                   Show this help message and exit\n\n"
          "Format of output table is tab-delimited with columns:\n"
          "Segment, IBD0_Score, IBD1_Score, IBD2_Score, Inferred_State\n",
          stderr);
    exit(code);
}

// "%.5Le" of exp(L): mantissa and exponent from the logarithm.
void put_score(char *dst, double L) {
    if (std::isnan(L)) {
        strcpy(dst, "-nan");
        return;
    }
    if (std::isinf(L) && L < 0) {
        strcpy(dst, "0.00000e+00");
        return;
    }
    const long double l10 = (long double)L / logl(10.0L);
    long double ex = floorl(l10);
    long double mant = powl(10.0L, l10 - ex);
    char m[32];
    snprintf(m, sizeof(m), "%.5Lf", mant);
    if (strncmp(m, "10.", 3) == 0) {  // rounded up to the next decade
        ex += 1;
        snprintf(m, sizeof(m), "%.5Lf", 1.0L);
    }
    const long e = (long)ex;
    sprintf(dst, "%se%c%02ld", m, e < 0 ? '-' : '+', e < 0 ? -e : e);
}

// fn(i) for i in [0, n) on up to eight threads (one when n == 1)
template <class F>
void parallel_for(size_t n, F fn) {
    const size_t nt = std::max<size_t>(1, std::min<size_t>({n, 8, (size_t)std::thread::hardware_concurrency()}));
    if (nt == 1) {
        for (size_t i = 0; i < n; i++) fn(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::vector<std::thread> pool;
    for (size_t k = 0; k < nt; k++)
        pool.emplace_back([&] {
            for (size_t i; (i = next.fetch_add(1)) < n;) fn(i);
        });
    for (auto &t : pool) t.join();
}

// init_summary, src/hiddengem.c:51-84: skip leading '#' lines, then every line that parses
// (START, END and NUM_SITES of each bin are kept for --tracts)
struct Summary {
    std::vector<double> lik;
    std::vector<uint64_t> start, end;
    std::vector<int64_t> n_sites;
};
int read_summary(const std::string &fn, Summary *sm) {
    LineReader lr;
    if (!lr.open(fn)) return 1;
    const char *line;
    size_t len;
    std::string z;
    bool body = false;
    while (lr.next(&line, &len)) {
        if (!body && len && line[0] == '#') continue;
        body = true;
        z.assign(line, len);
        size_t a, b;
        double l0, l1, l2;
        int n;
        if (sscanf(z.c_str(), "%*s\t%zu\t%zu\t%lf\t%lf\t%lf\t%d", &a, &b, &l0, &l1, &l2, &n) == 6) {
            sm->lik.push_back(l0);
            sm->lik.push_back(l1);
            sm->lik.push_back(l2);
            sm->start.push_back(a);
            sm->end.push_back(b);
            sm->n_sites.push_back(n);
        }
    }
    return 0;
}

}  // namespace

int main(int argc, char *argv[]) {
    double p01 = 0.001, p02 = 0.000001, p12 = 0.001;
    std::vector<std::string> files;
    bool posterior = false, share_sd = false, tract_counts = false, tract_lengths = false, lengths_ok = true;
    std::vector<uint64_t> thresholds;  // --tract-lengths
    const char *tracts_fn = nullptr;
    static struct option longopts[] = {{"summary", required_argument, 0, 's'}, {"p01", required_argument, 0, 1},
                                       {"p02", required_argument, 0, 2},       {"p12", required_argument, 0, 3},
                                       {"posterior", no_argument, 0, 4},       // additive
                                       {"tracts", required_argument, 0, 5},    // additive
                                       {"share-sd", no_argument, 0, 6},        // additive
                                       {"tract-counts", no_argument, 0, 7},    // additive
                                       {"tract-lengths", required_argument, 0, 8},  // additive
                                       {"help", no_argument, 0, 'h'},          {0, 0, 0, 0}};
    if (argc == 1) print_help(0);
    int option;
    while ((option = getopt_long(argc, argv, ":s:h", longopts, nullptr)) != -1) {
        switch (option) {
            case 's': files.push_back(optarg); break;
            case 1: p01 = atof(optarg); break;
            case 2: p02 = atof(optarg); break;
            case 3: p12 = atof(optarg); break;
            case 4: posterior = true; break;
            case 5: tracts_fn = optarg; break;
            case 6: share_sd = true; break;
            case 7: tract_counts = true; break;
            case 8:
                tract_lengths = true;
                lengths_ok = parse_tract_lengths(optarg, &thresholds);
                break;
            case 'h': print_help(0); break;
            case ':':
                fprintf(stderr, "Option -%c missing required argument.\n", optopt);
                exit(0);
            case '?':
                if (isprint(optopt)) fprintf(stderr, "Invalid option -%c.\n", optopt);
                else fprintf(stderr, "Invalid option character.\n");
                break;
            default:
                fprintf(stderr, "[::] ERROR parsing command-line options.\n");
                exit(0);
        }
    }
    for (int i = optind; i < argc; i++) fprintf(stderr, "Given extra argument %s.\n", argv[i]);
    if (share_sd && !posterior) {
        fprintf(stderr, "[::] ERROR: --share-sd needs --posterior (the standard deviations are those of the posterior counts).\n");
        exit(0);
    }
    if (tract_counts && !posterior) {
        fprintf(stderr, "[::] ERROR: --tract-counts needs --posterior (the tract counts are those of the posterior paths).\n");
        exit(0);
    }
    if (tract_lengths && !posterior) {
        fprintf(stderr, "[::] ERROR: --tract-lengths needs --posterior (the run lengths are those of the posterior paths).\n");
        exit(0);
    }
    if (tract_lengths && !lengths_ok) {
        fputs(kTractLengthsError, stderr);
        exit(0);
    }

    // the tables are independent files: read by a few threads, concatenated in command-line order
    std::vector<Summary> per_file(files.size());
    std::vector<int> read_rc(files.size(), 0);
    parallel_for(files.size(), [&](size_t i) { read_rc[i] = read_summary(files[i], &per_file[i]); });
    std::vector<double> lik;
    std::vector<int64_t> off{0};
    for (size_t i = 0; i < files.size(); i++) {
        if (read_rc[i]) exit(1);
        lik.insert(lik.end(), per_file[i].lik.begin(), per_file[i].lik.end());
        std::vector<double>().swap(per_file[i].lik);
        off.push_back((int64_t)(lik.size() / 3));
    }
    if (files.empty() || lik.empty()) {
        fprintf(stderr, "[::] ERROR parsing likelihood data; make sure input is valid.\n");
        exit(1);
    }
    const size_t nb = lik.size() / 3;
    ibdgem_params prm{};
    prm.epsilon = 0.02; prm.max_cov = 20; prm.window_size = 100; prm.min_af = 0; prm.max_af = 1;
    ibdgem_engine *e = nullptr;
    std::vector<uint8_t> state(nb);
    std::vector<double> score(nb * 3);
    std::vector<int64_t> counts((off.size() - 1) * 3);
    std::vector<double> post(posterior ? nb * 3 : 0), expected(posterior ? (off.size() - 1) * 3 : 0);
    std::vector<double> cov(share_sd ? (off.size() - 1) * 9 : 0);
    const size_t ntc = tract_counts ? off.size() - 1 : 0;  // --tract-counts: expected (again), switches, tracts, tract_cov
    std::vector<double> tc_expected(ntc * 3), tc_switches(ntc * 9), tc_tracts(ntc * 3), tc_cov(ntc * 9);
    const size_t nk = thresholds.size();  // --tract-lengths: the spectrum on the START / END columns
    std::vector<double> spectrum((tract_lengths ? off.size() - 1 : 0) * nk * 3);
    std::vector<uint64_t> bin_start, bin_end;
    for (size_t i = 0; tract_lengths && i < files.size(); i++) {
        bin_start.insert(bin_start.end(), per_file[i].start.begin(), per_file[i].start.end());
        bin_end.insert(bin_end.end(), per_file[i].end.begin(), per_file[i].end.end());
    }
    if (ibdgem_engine_create(&prm, &e) ||
        hiddengem_viterbi_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, state.data(), score.data(),
                                counts.data()) ||
        (posterior && !share_sd &&
         hiddengem_posterior_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, post.data(), expected.data())) ||
        (share_sd && hiddengem_posterior_moments_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, post.data(),
                                                       expected.data(), cov.data())) ||
        (tract_counts && hiddengem_tract_counts_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, tc_expected.data(),
                                                      tc_switches.data(), tc_tracts.data(), tc_cov.data())) ||
        (tract_lengths && hiddengem_tract_lengths_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, bin_start.data(),
                                                        bin_end.data(), (int32_t)nk, thresholds.data(), spectrum.data()))) {
        fprintf(stderr, "%s\n", ibdgem_last_error());
        exit(1);
    }
    if (tracts_fn) {  // the same tables once more, through the tract entry: only the records come back
        std::vector<int64_t> toff(off.size());
        std::vector<hiddengem_tract> tr;
        int rc = hiddengem_tracts_batch(e, (int32_t)off.size() - 1, off.data(), lik.data(), 0, p01, p02, p12, posterior ? 1 : 0, toff.data());
        if (!rc) {
            tr.resize((size_t)toff.back());
            rc = hiddengem_last_tracts(e, tr.data(), 0);
        }
        if (rc) {
            fprintf(stderr, "%s\n", ibdgem_last_error());
            exit(1);
        }
        FILE *f = fopen(tracts_fn, "w");
        if (!f) {
            fprintf(stderr, "[::] ERROR: Cannot open '%s' for writing.\n", tracts_fn);
            exit(1);
        }
        const std::string head = tract_header(true, posterior);
        fwrite(head.data(), 1, head.size(), f);
        for (size_t t = 0; t + 1 < off.size(); t++) {
            const Summary &sm = per_file[t];
            for (int64_t k = toff[t]; k < toff[t + 1]; k++) {
                const hiddengem_tract &r = tr[(size_t)k];
                const size_t a = (size_t)r.first_bin, b = (size_t)(r.first_bin + r.n_bins);
                int64_t sites = 0;
                for (size_t i = a; i < b; i++) sites += sm.n_sites[i];
                const std::string row = files[t] + "\t" + tract_row(r, k - toff[t], sm.start[a], sm.end[b - 1], sites, posterior);
                fwrite(row.data(), 1, row.size(), f);
            }
        }
        if (fclose(f)) {
            fprintf(stderr, "[::] ERROR: Cannot write '%s'.\n", tracts_fn);
            exit(1);
        }
    }
    ibdgem_engine_destroy(e);
    // one table's text does not depend on another's: formatted by a few threads, a wave of tables at a
    // time, written in order
    const size_t n_tables = off.size() - 1, wave = 64;
    std::vector<std::string> text(wave);
    for (size_t t0 = 0; t0 < n_tables; t0 += wave) {
        const size_t nt = std::min(wave, n_tables - t0);
        parallel_for(nt, [&](size_t k) {
            const size_t t = t0 + k;
            const int64_t a = off[t], b = off[t + 1];
            const double n = (double)(b - a);
            std::string &out = text[k];
            out.clear();
            out.reserve((size_t)(b - a) * (posterior ? 80 : 48) + 512);
            out += posterior ? "Segment\tIBD0_Score\tIBD1_Score\tIBD2_Score\tInferred_State\tP_IBD0\tP_IBD1\tP_IBD2\n"
                             : "Segment\tIBD0_Score\tIBD1_Score\tIBD2_Score\tInferred_State\n";
            char s0[48], s1[48], s2[48], row[192];
            for (int64_t i = a; i < b; i++) {
                put_score(s0, score[(size_t)i * 3]);
                put_score(s1, score[(size_t)i * 3 + 1]);
                put_score(s2, score[(size_t)i * 3 + 2]);
                if (posterior)
                    out.append(row, (size_t)snprintf(row, sizeof row, "%d\t%s\t%s\t%s\t%d\t%.6f\t%.6f\t%.6f\n", (int)(i - a + 1), s0, s1, s2,
                                                     (int)state[(size_t)i], post[(size_t)i * 3], post[(size_t)i * 3 + 1], post[(size_t)i * 3 + 2]));
                else
                    out.append(row, (size_t)snprintf(row, sizeof row, "%d\t%s\t%s\t%s\t%d\n", (int)(i - a + 1), s0, s1, s2, (int)state[(size_t)i]));
            }
            const double c0 = (double)counts[t * 3], c1 = (double)counts[t * 3 + 1], c2 = (double)counts[t * 3 + 2];
            out.append(row, (size_t)snprintf(row, sizeof row, "#%% IBD0 (n = %.0f): %.2f\n", c0, (c0 / n) * 100));
            out.append(row, (size_t)snprintf(row, sizeof row, "#%% IBD1 (n = %.0f): %.2f\n", c1, (c1 / n) * 100));
            out.append(row, (size_t)snprintf(row, sizeof row, "#%% IBD2 (n = %.0f): %.2f\n", c2, (c2 / n) * 100));
            if (posterior)  // expected bins per state: the sum of the posteriors
                for (int k = 0; k < 3; k++) {
                    const double x = expected[t * 3 + (size_t)k];
                    out.append(row, (size_t)snprintf(row, sizeof row, "#%% posterior IBD%d (n = %.2f): %.2f\n", k, x, (x / n) * 100));
                }
            if (share_sd) out += share_sd_lines(&expected[t * 3], &cov[t * 9], n);
            if (tract_counts) out += tract_count_lines(&tc_tracts[t * 3], &tc_cov[t * 9], &tc_switches[t * 9]);
            if (tract_lengths) out += tract_length_lines(&spectrum[t * nk * 3], thresholds);
        });
        for (size_t k = 0; k < nt; k++) fwrite(text[k].data(), 1, text[k].size(), stdout);
    }
    if ((share_sd || tract_counts || tract_lengths) && n_tables > 1) {  // the tables are independent: their means and covariances add
        double x[3] = {0, 0, 0}, c[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        std::vector<double> sp(nk * 3, 0.0);
        double tt[3] = {0, 0, 0}, tcv[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, sw[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (size_t t = 0; t < n_tables; t++) {
            for (int k = 0; k < 3; k++) x[k] += expected[t * 3 + (size_t)k];
            for (int k = 0; k < 9 && share_sd; k++) c[k] += cov[t * 9 + (size_t)k];
            for (int k = 0; k < 3 && tract_counts; k++) tt[k] += tc_tracts[t * 3 + (size_t)k];
            for (int k = 0; k < 9 && tract_counts; k++) {
                tcv[k] += tc_cov[t * 9 + (size_t)k];
                sw[k] += tc_switches[t * 9 + (size_t)k];
            }
            for (size_t k = 0; k < nk * 3 && tract_lengths; k++) sp[k] += spectrum[t * nk * 3 + k];
        }
        const double n = (double)off.back();
        std::string out;
        char row[160];
        out.append(row, (size_t)snprintf(row, sizeof row, "#%% all %zu tables (n = %.0f)\n", n_tables, n));
        for (int k = 0; k < 3; k++)
            out.append(row, (size_t)snprintf(row, sizeof row, "#%% posterior IBD%d (n = %.2f): %.2f\n", k, x[k], (x[k] / n) * 100));
        if (share_sd) out += share_sd_lines(x, c, n);
        if (tract_counts) out += tract_count_lines(tt, tcv, sw);
        if (tract_lengths) out += tract_length_lines(sp.data(), thresholds);
        fwrite(out.data(), 1, out.size(), stdout);
    }
    return 0;
}
