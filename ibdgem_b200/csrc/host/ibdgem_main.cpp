// ibdgem — command-line front-end of the B200-native engine.  Same options, defaults, messages,
// exit codes and output tables as the reference's main()/compare_impute()/compare_vcf()
// (src/ibdgem.c:41-66, 779-1183); the arithmetic is done by libibdgem_b200.so through the C ABI
// (include/ibdgem_b200.h) and there is no CPU fallback.  Additive options: --gpus N (shard the
// targets over N devices), --batch N (targets per engine call), --no-tab (skip *.tab.txt),
// --panel-cache FILE (binary cache of the parsed IMPUTE or VCF panel), --hiddengem [--p01/--p02/--p12] (chain the
// batched Viterbi pass over each target's window scores: <pileup>.<target>.hiddengem.txt; with --tracts also the IBD
// tracts, maximal runs of one state, in <pileup>.<target>.tracts.txt).
#include <getopt.h>
#include <limits.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "../../../include/ibdgem_b200.h"
#include "panel.h"
#include "pileup_store.h"
#include "textio.h"

using namespace ibdhost;

namespace {

struct Options {
    double epsilon = 0.02, min_qual = 0, max_af = 1, min_af = 0, target_dp = 0;
    unsigned max_cov = 20;
    int window = 100;
    const char *sq_id = "UNKWN";
    int ld = 0, in_impute = 0, in_vcf = 0, opt_s1 = 0, opt_s2 = 0, opt_b = 0, opt_a = 0, opt_p = 0, opt_v = 0, opt_d = 0;
    std::string vcf_fn, hap_fn, legend_fn, indv_fn, pu_fn, sample_fn, ref_fn, af_fn, pos_fn, sample_str, out_dir;
    std::string cache_fn;  // --panel-cache
    const char *uchr = nullptr;
    int gpus = 1, batch = 0, no_tab = 0;
    int hiddengem = 0;  // --hiddengem: also write <pileup>.<target>.hiddengem.txt from the window scores
    int posterior = 0;  // --posterior (with --hiddengem): posterior state probabilities in those files
    int tracts = 0;     // --tracts (with --hiddengem): also write <pileup>.<target>.tracts.txt
    int share_sd = 0;   // --share-sd (with --posterior): sd of the posterior state shares and kinship in those files
    double p01 = 0.001, p02 = 0.000001, p12 = 0.001;
};

void print_help(int code) {
    static const char *const kHelp =
        "IBDGem-2.0: Compares low-coverage sequencing data from an unknown sample to known genotypes\n"
        "            from a reference individual/panel and calculates the likelihood that the samples\n"
        "            share 0, 1, or 2 IBD chromosomes.\n\n"
        "Usage: ./ibdgem [--LD] -H [hap-file] -L [legend-file] -I [indv-file] -P [pileup-file] [other options...]\n"
        "       OR ./ibdgem [--LD] -V [vcf-file] -P [pileup-file] [other options...]\n"
        "--LD                            Linkage disequilibrium mode ON (default: OFF)\n"
        "-V, --vcf  FILE                 VCF file (required if using VCF)\n"
        "-H, --hap  FILE                 HAP file (required if using IMPUTE)\n"
        "-L, --legend  FILE              LEGEND file (required if using IMPUTE)\n"
        "-I, --indv  FILE                INDV file (required if using IMPUTE)\n"
        "-P, --pileup  FILE              PILEUP file (required)\n"
        "-N, --pileup-name  STR          Name of Pileup sample (default: UNKWN)\n"
        "-A, --allele-freqs  FILE        File containing allele frequencies from a background panel;\n"
        "                                   must be sorted & whitespace-delimited with columns CHROM, POS, AF;\n"
        "                                   use in conjunction with -c if includes multiple chromosomes\n"
        "                                   (default: calculate AF from input genotypes)\n"
        "-S, --sample-list  FILE         File containing subset of samples to compare the\n"
        "                                   sequencing data against; one line per sample\n"
        "                                   (default: compare against all samples in genotype file)\n"
        "-s, --sample  STR               Sample(s) to compare the sequencing data against; comma-separated\n"
        "                                   without spaces if more than one (e.g. sample1,sample2,etc.)\n"
        "-B, --background-list  FILE     File containing subset of samples to be used as the background panel\n"
        "                                   for calculating IBD0 and IBD1 in LD mode; one line per sample\n"
        "                                   (default: use all samples in genotype file as background)\n"
        "-p, --positions  FILE           List of sites to compare; can be in position list format with 2 columns\n"
        "                                   CHROM, POS (1-based coordinates) or BED format (0-based coordinates);\n"
        "                                   use in conjunction with -c if includes multiple chromosomes\n"
        "                                   (default: perform comparison at all sites)\n"
        "-q, --min-qual  FLOAT           Genotype quality minimum when using VCF input (default: no minimum)\n"
        "-M, --max-cov  INT              Maximum estimated coverage of Pileup data (default: 20)\n"
        "-F, --max-af  FLOAT             Maximum alternate allele frequency (default: 1)\n"
        "-f, --min-af  FLOAT             Minimum alternate allele frequency (default: 0)\n"
        "-D, --downsample-cov  FLOAT     Down-sample to this fold-coverage depth\n"
        "-w, --window-size  INT          Number of sites per genomic segment over which likelihood results\n"
        "                                   are summarized/aggregated (default: 100)\n"
        "-O, --out-dir  STR              Path to output directory (default: output to current directory)\n"
        "-c, --chromosome  STR           Chromosome on which the comparison is done; if not specified,\n"
        "                                   will assume that all inputs are on one single chromosome\n"
        "-e, --error-rate  FLOAT         Error rate of sequencing platform (default: 0.02)\n"
        "-v, --variable-sites-only       If set, make output only for sites that are not\n"
        "                                   homozygous reference in the genotype file for this sample\n"
        "--hiddengem                     Also infer IBD states from each target's window scores: writes\n"
        "                                   <pileup-name>.<target>.hiddengem.txt (penalties --p01, --p02, --p12)\n"
        "--posterior                     With --hiddengem: add each segment's posterior state probabilities\n"
        "                                   (P_IBD0, P_IBD1, P_IBD2) and the expected share of segments per state\n"
        "--share-sd                      With --posterior: add the standard deviation of each state's share of\n"
        "                                   segments and the window-share kinship (N_IBD1/4 + N_IBD2/2)/n with\n"
        "                                   its standard deviation, from the posterior covariance\n"
        "--tracts                        With --hiddengem: also write the IBD tracts (maximal runs of segments in\n"
        "                                   one state) to <pileup-name>.<target>.tracts.txt: state, first and last\n"
        "                                   segment, START, END, number of segments and sites, LOD10 of the state\n"
        "                                   against the next best (and with --posterior its mean and minimum posterior)\n"
        "-h, --help                      Show this help message and exit\n\n"
        "Format of likelihood table is tab-delimited with columns:\n"
        "CHR, rsID, POS, REF, ALT, AF, DP, SQ_NREF, SQ_NALT, GT_A0, GT_A1, LIBD0, LIBD1, LIBD2\n\n"
        "Format of summary file is tab-delimited with columns:\n"
        "SEGMENT, START, END, LIBD0, LIBD1, LIBD2, NUM_SITES\n";
    fputs(kHelp, stderr);
    exit(code);
}

// C's %e of a double, with the reference's "-nan" for 0/0 (src/ibdgem.c:751-752)
// "%.5Le" of exp(L) from its logarithm (hiddengem's score columns; same routine as hiddengem_main.cpp)
void put_score_log(char *dst, double L) {
    if (std::isnan(L)) { strcpy(dst, "-nan"); return; }
    if (std::isinf(L) && L < 0) { strcpy(dst, "0.00000e+00"); return; }
    const long double l10 = (long double)L / logl(10.0L);
    long double ex = floorl(l10);
    long double mant = powl(10.0L, l10 - ex);
    char m[32];
    snprintf(m, sizeof(m), "%.5Lf", mant);
    if (strncmp(m, "10.", 3) == 0) {
        ex += 1;
        snprintf(m, sizeof(m), "%.5Lf", 1.0L);
    }
    const long e = (long)ex;
    sprintf(dst, "%se%c%02ld", m, e < 0 ? '-' : '+', e < 0 ? -e : e);
}

int put_e(char *dst, double v) {
    if (std::isnan(v)) return sprintf(dst, "-nan");
    return sprintf(dst, "%e", v);
}

struct InputDist {
    std::vector<unsigned long> dist;
    double mean = 0, cull_p = 1;
};

// find_cull_p, src/ibdgem.c:83-106
InputDist input_distribution(const PileupStore &pu, const Options &o) {
    InputDist d;
    d.dist.assign(o.max_cov + 1, 0);
    unsigned long total = 0;
    for (size_t i = 0; i < pu.size(); i++)
        if (pu.cov[i] <= o.max_cov) {
            total += pu.cov[i];
            d.dist[pu.cov[i]]++;
        }
    d.mean = (double)total / pu.size();
    if (o.opt_d) {
        if (o.target_dp > d.mean) fprintf(stderr, "Observed depth is lower than target depth -D. No culling will be done.\n");
        else d.cull_p = o.target_dp / d.mean;
    }
    return d;
}

struct Shared {
    const Options *opt;
    const PackedPanel *panel;
    const PileupStore *pu;
    const InputDist *dist;
    std::string user_cmd;
    std::vector<Sample> targets, background;
    int pu_idx = -1;
    std::vector<uint8_t> tgt_counts;  // -D: [T][S][2], drawn in reference order
    int rc = 0;
};

constexpr int WRITER_THREADS = 8;  // per device shard

// Per-site text of the tab.txt rows for runs without -D: the row prefix
// "CHR\trsID\tPOS\tREF\tALT\tAF\tDP\tSQ_NREF\tSQ_NALT\t" and the seven likelihood strings a row can
// show (LIBD0; LIBD1 and LIBD2 for g = 0, 1, 2), formatted with the C library exactly as a row-by-row
// writer would (src/ibdgem.c:731-733).  A row is then two allele digits between copies of these.
struct SiteText {
    static constexpr size_t NONE = ~(size_t)0;
    std::vector<size_t> off;   // offset of the site's record in `blob`, NONE if the site prints no row
    std::vector<char> blob;    // record: u16 prefix length, prefix bytes, 7 x (u8 length, 15 bytes)
    bool has(size_t s) const { return !off.empty() && off[s] != NONE; }
    void build(const PackedPanel &P, const PileupStore &pu, const std::vector<uint8_t> &status, const std::vector<double> &f,
               const std::vector<double> &lik7) {
        const size_t S = (size_t)P.S;
        off.assign(S, NONE);
        std::vector<char> tmp(1 << 12);
        for (size_t s = 0; s < S; s++) {
            if (!status[s]) continue;
            const std::string &chr = pu.chr_names[P.chr_id[s]];
            if (tmp.size() < chr.size() + P.id_len[s] + 256) tmp.resize(chr.size() + P.id_len[s] + 256);
            char *q = tmp.data();
            memcpy(q, chr.data(), chr.size()); q += chr.size();
            *q++ = '\t';
            memcpy(q, P.text.data() + P.id_off[s], P.id_len[s]); q += P.id_len[s];
            q += sprintf(q, "\t%lu\t%c\t%c\t%lf\t%u\t%u\t%u\t", (unsigned long)P.pos[s], P.ref[s], P.alt[s], f[s], P.dp[s],
                         (unsigned)P.n_ref[s], (unsigned)P.n_alt[s]);
            const size_t plen = (size_t)(q - tmp.data());
            if (plen > 0xFFFF) continue;  // (a 64 KB rsID: leave the row to the generic writer)
            off[s] = blob.size();
            const uint16_t plen16 = (uint16_t)plen;
            blob.insert(blob.end(), reinterpret_cast<const char *>(&plen16), reinterpret_cast<const char *>(&plen16) + 2);
            blob.insert(blob.end(), tmp.data(), tmp.data() + plen);
            for (int j = 0; j < 7; j++) {
                char e[40];
                const int n = put_e(e, lik7[s * 7 + (size_t)j]);
                char slot[16] = {0};
                slot[0] = (char)n;  // "%e" of a double is at most 14 characters
                memcpy(slot + 1, e, (size_t)n);
                blob.insert(blob.end(), slot, slot + 16);
            }
        }
    }
    // writes the whole row of site s for a target with alleles a0, a1 (g = a0 + a1); returns the end
    char *put_row(char *q, size_t s, unsigned a0, unsigned a1, unsigned g) const {
        const char *r = blob.data() + off[s];
        uint16_t plen;
        memcpy(&plen, r, 2);
        memcpy(q, r + 2, plen); q += plen;
        *q++ = (char)('0' + a0); *q++ = '\t';
        *q++ = (char)('0' + a1); *q++ = '\t';
        const char *slots = r + 2 + plen;
        const int pick[3] = {0, 1 + (int)g, 4 + (int)g};
        for (int j = 0; j < 3; j++) {
            const char *sl = slots + 16 * pick[j];
            memcpy(q, sl + 1, 15);  // fixed-size copy, advance by the real length
            q += (unsigned char)sl[0];
            *q++ = j == 2 ? '\n' : '\t';
        }
        return q;
    }
};

int fail_engine() {
    fprintf(stderr, "%s\n", ibdgem_last_error());
    return 1;
}

// Scores targets [t0, t1) on one device and writes their two tables.
// --gpus N: device 0's engine is the one that uploads the panel over PCIe; the others clone it over NVLink
// (ibdgem_engine_clone_panel) as its chunks land.  The engine pointer is published once its upload has been issued.
struct PanelSource {
    std::mutex mu;
    std::condition_variable cv;
    ibdgem_engine *engine = nullptr;
    bool failed = false;
    std::atomic<int> users{0};  // clones still reading from it
};

int run_shard(Shared *sh, int device, size_t t0, size_t t1, PanelSource *psrc = nullptr) {
    const Options &o = *sh->opt;
    const PackedPanel &P = *sh->panel;
    const size_t S = (size_t)P.S;
    ibdgem_params prm{};
    prm.epsilon = o.epsilon;
    prm.max_cov = o.max_cov;
    prm.window_size = o.window;
    prm.min_af = o.min_af;
    prm.max_af = o.max_af;
    prm.variable_sites_only = o.opt_v;
    prm.device = device;
    ibdgem_engine *e = nullptr;
    struct Release {  // a clone stops reading the source engine's panel at the latest when its shard is done (any exit path)
        PanelSource *p;
        ~Release() { if (p) p->users.fetch_sub(1); }
    } release{psrc && device != 0 ? psrc : nullptr};
    struct Publish {  // device 0 leaving before it has published its engine must not leave the clones waiting
        PanelSource *p;
        bool done = false;
        ~Publish() {
            if (p && !done) {
                std::lock_guard<std::mutex> lk(p->mu);
                p->failed = true;
                p->cv.notify_all();
            }
        }
    } publish{psrc && device == 0 ? psrc : nullptr};
    if (ibdgem_engine_create(&prm, &e)) return fail_engine();
    if (ibdgem_engine_upload_sites(e, P.S, P.pos.data(), P.n_ref.data(), P.n_alt.data(), P.host_keep.data(),
                                   P.af_user.empty() ? nullptr : P.af_user.data()))
        return fail_engine();
    if (psrc && device != 0) {
        std::unique_lock<std::mutex> lk(psrc->mu);
        psrc->cv.wait(lk, [&] { return psrc->engine || psrc->failed; });
        if (psrc->failed) return 1;
        if (ibdgem_engine_clone_panel(e, psrc->engine)) return fail_engine();
    } else {
        const int urc = ibdgem_engine_upload_panel(e, P.S, P.N, P.bits.data(), P.Wh);
        if (psrc) {
            std::lock_guard<std::mutex> lk(psrc->mu);
            psrc->engine = urc ? nullptr : e;
            psrc->failed = urc != 0;
            psrc->cv.notify_all();
            publish.done = true;
        }
        if (urc) return fail_engine();
    }
    if (ibdgem_engine_prepare(e)) return fail_engine();

    std::vector<double> f(S), lik7(S * 7);
    std::vector<uint8_t> st_shared(S);
    if (ibdgem_engine_get_site_table(e, f.data(), st_shared.data(), lik7.data())) return fail_engine();

    const bool per_target = o.opt_v || sh->dist->cull_p != 1.0;  // kept set / counts depend on the target
    const bool culled = sh->dist->cull_p != 1.0;
    const int C = (int)o.max_cov + 1;
    const int maxW = (int)(S / (size_t)o.window + 2);
    size_t batch = o.batch > 0 ? (size_t)o.batch : 256;
    if (per_target) batch = std::min<size_t>(batch, std::max<size_t>(1, ((size_t)1 << 30) / (S * 25 + 1)));
    std::vector<int32_t> bg(sh->background.size());
    for (size_t i = 0; i < bg.size(); i++) bg[i] = sh->background[i].ordinal;

    // Everything a tab.txt row says besides the target's two alleles depends on the site alone (and, for
    // the likelihoods, on the genotype class g): format it once per site, not once per target and site
    // (SURVEY.md 8f-2: 1,000 targets x 1 M rows is 100 GB of text).  -D makes counts and likelihoods
    // target-dependent; those runs format row by row.
    SiteText site_text;
    if (!o.no_tab && !culled) site_text.build(P, *sh->pu, st_shared, f, lik7);

    for (size_t b0 = t0; b0 < t1; b0 += batch) {
        const size_t T = std::min(batch, t1 - b0);
        std::vector<int32_t> tg(T);
        for (size_t k = 0; k < T; k++) tg[k] = sh->targets[b0 + k].ordinal;
        std::vector<int32_t> nw(T), wn(T * (size_t)maxW);
        std::vector<uint64_t> ws(T * (size_t)maxW), we(T * (size_t)maxW), processed(T), skipped(T), totcov(T), fdist(T * (size_t)C);
        std::vector<double> wll(T * (size_t)maxW * 3);
        // the reference's own linear window products (bit for bit, underflow included): the three columns of a non-LD
        // summary row and LIBD2 of an --LD row are printed from them, so those columns are the reference's bytes
        const bool want_linear = !(o.ld && per_target);
        std::vector<double> wlin(want_linear ? T * (size_t)maxW * 3 : 0);
        std::vector<uint8_t> sst;
        std::vector<double> slik;
        ibdgem_scores sc{};
        sc.max_windows = maxW;
        sc.n_windows = nw.data(); sc.w_start = ws.data(); sc.w_end = we.data(); sc.w_nsites = wn.data();
        sc.w_loglik = wll.data(); sc.processed = processed.data(); sc.skipped = skipped.data();
        sc.final_total_cov = totcov.data(); sc.final_dist = fdist.data();
        if (want_linear) sc.w_lik_linear = wlin.data();
        if (per_target) {
            sst.resize(T * S);
            sc.site_status = sst.data();
            if (culled) {
                slik.resize(T * S * 3);
                sc.site_lik = slik.data();
            }
        }
        const uint8_t *tc = culled ? sh->tgt_counts.data() + b0 * S * 2 : nullptr;
        const int rc = o.ld ? ibdgem_engine_score_ld(e, (int32_t)T, tg.data(), (int32_t)bg.size(), bg.data(), sh->pu_idx, tc, &sc)
                            : ibdgem_engine_score_nonld(e, (int32_t)T, tg.data(), tc, &sc);
        if (rc) return fail_engine();

        for (size_t k = 0; k < T; k++)
            fprintf(stderr, "Running %s-vs-%s comparison...\n", o.sq_id, sh->targets[b0 + k].name.c_str());

        // --hiddengem: the batch's window scores go straight into the batched Viterbi as natural logs (is_log = 1) —
        // no round trip through the 7-digit text of summary.txt that the reference's hiddengem parses
        // (src/hiddengem.c:66-76).  One table per target, in the same call order.
        std::vector<uint8_t> hg_state;
        std::vector<double> hg_score;
        std::vector<int64_t> hg_counts, hg_off;
        std::vector<double> hg_post, hg_expected, hg_cov;
        std::vector<int64_t> tr_off;
        std::vector<hiddengem_tract> tracts;
        if (o.hiddengem) {
            std::vector<double> packed;
            hg_off.assign(1, 0);
            for (size_t k = 0; k < T; k++) {
                packed.insert(packed.end(), wll.begin() + (ptrdiff_t)(k * (size_t)maxW * 3), wll.begin() + (ptrdiff_t)((k * (size_t)maxW + (size_t)nw[k]) * 3));
                hg_off.push_back(hg_off.back() + nw[k]);
            }
            const size_t nbins = (size_t)hg_off.back();
            hg_state.resize(nbins);
            hg_score.resize(nbins * 3);
            hg_counts.resize(T * 3);
            if (nbins && hiddengem_viterbi_batch(e, (int32_t)T, hg_off.data(), packed.data(), 1, o.p01, o.p02, o.p12, hg_state.data(),
                                                 hg_score.data(), hg_counts.data()))
                return fail_engine();
            if (o.posterior) {  // the same packed natural-log scores
                hg_post.resize(nbins * 3);
                hg_expected.resize(T * 3);
                if (!o.share_sd && nbins &&
                    hiddengem_posterior_batch(e, (int32_t)T, hg_off.data(), packed.data(), 1, o.p01, o.p02, o.p12, hg_post.data(), hg_expected.data()))
                    return fail_engine();
                hg_cov.resize(o.share_sd ? T * 9 : 0);
                if (o.share_sd && nbins &&
                    hiddengem_posterior_moments_batch(e, (int32_t)T, hg_off.data(), packed.data(), 1, o.p01, o.p02, o.p12, hg_post.data(),
                                                      hg_expected.data(), hg_cov.data()))
                    return fail_engine();
            }
            if (o.tracts && nbins) {  // the same packed scores through the tract entry: only the records come back
                tr_off.resize(T + 1);
                if (hiddengem_tracts_batch(e, (int32_t)T, hg_off.data(), packed.data(), 1, o.p01, o.p02, o.p12, o.posterior, tr_off.data()))
                    return fail_engine();
                tracts.resize((size_t)tr_off[T]);
                if (hiddengem_last_tracts(e, tracts.data(), 0)) return fail_engine();
            }
        }

        // one target = two files: independent, so the batch is written by a few threads
        auto write_target = [&](size_t k, std::vector<char> &line) -> int {
            const Sample &smp = sh->targets[b0 + k];
            const std::string tab_fn = o.out_dir + "/" + o.sq_id + "." + smp.name + ".tab.txt";
            const std::string sum_fn = o.out_dir + "/" + o.sq_id + "." + smp.name + ".summary.txt";
            FILE *tab = o.no_tab ? nullptr : fopen(tab_fn.c_str(), "w");
            FILE *sum = fopen(sum_fn.c_str(), "w");
            if ((!o.no_tab && !tab) || !sum) {
                fprintf(stderr, "[::] ERROR in compare_%s(): Cannot open '%s' and/or '%s' for writing.\n", o.in_vcf ? "vcf" : "impute",
                        tab_fn.c_str(), sum_fn.c_str());
                if (tab) fclose(tab);
                if (sum) fclose(sum);
                return 1;
            }
            if (tab) {
                setvbuf(tab, nullptr, _IOFBF, 1 << 20);
                fprintf(tab, "# Entered command: %s\n\n", sh->user_cmd.c_str());
                fprintf(tab, "# INPUT COVERAGE DISTRIBUTION:\n# COVERAGE N_SITES\n");
                for (unsigned c = 0; c <= o.max_cov; c++) fprintf(tab, "# %d %lu\n", (int)c, sh->dist->dist[c]);
                fprintf(tab, "# MEAN DEPTH = %lf\n# CULL DEPTH RATIO = %lf\n", sh->dist->mean, sh->dist->cull_p);
                fprintf(tab, "# CHR\trsID\tPOS\tREF\tALT\tAF\tDP\tSQ_NREF\tSQ_NALT\tGT_A0\tGT_A1\tLIBD0\tLIBD1\tLIBD2\n");
                const size_t h0 = 2 * (size_t)smp.ordinal;
                size_t fill = 0;  // rows are gathered in `line` and written in large pieces
                for (size_t s = 0; s < S; s++) {
                    const uint8_t st = per_target ? sst[k * S + s] : st_shared[s];
                    if (!st) continue;
                    const uint32_t *row = P.bits.data() + s * (size_t)P.Wh;
                    const unsigned a0 = (row[h0 >> 5] >> (h0 & 31)) & 1u, a1 = (row[(h0 + 1) >> 5] >> ((h0 + 1) & 31)) & 1u;
                    const unsigned g = a0 + a1;
                    const std::string &chr = sh->pu->chr_names[P.chr_id[s]];
                    const size_t need = chr.size() + P.id_len[s] + 512;
                    if (line.size() < fill + need) {
                        if (fill) fwrite(line.data(), 1, fill, tab);
                        fill = 0;
                        if (line.size() < need) line.resize(need);
                    }
                    char *q = line.data() + fill;
                    if (site_text.has(s)) {
                        q = site_text.put_row(q, s, a0, a1, g);
                    } else {
                        double l0, l1, l2;
                        unsigned nr = P.n_ref[s], na = P.n_alt[s];
                        if (culled) {
                            l0 = slik[(k * S + s) * 3]; l1 = slik[(k * S + s) * 3 + 1]; l2 = slik[(k * S + s) * 3 + 2];
                            nr = tc[(k * S + s) * 2];
                            na = tc[(k * S + s) * 2 + 1];
                        } else {
                            l0 = lik7[s * 7]; l1 = lik7[s * 7 + 1 + g]; l2 = lik7[s * 7 + 4 + g];
                        }
                        memcpy(q, chr.data(), chr.size()); q += chr.size();
                        *q++ = '\t';
                        memcpy(q, P.text.data() + P.id_off[s], P.id_len[s]); q += P.id_len[s];
                        q += sprintf(q, "\t%lu\t%c\t%c\t%lf\t%u\t%u\t%u\t%u\t%u\t", (unsigned long)P.pos[s], P.ref[s], P.alt[s], f[s],
                                     P.dp[s], nr, na, a0, a1);
                        q += put_e(q, l0); *q++ = '\t';
                        q += put_e(q, l1); *q++ = '\t';
                        q += put_e(q, l2); *q++ = '\n';
                    }
                    fill = (size_t)(q - line.data());
                }
                if (fill) fwrite(line.data(), 1, fill, tab);
                fprintf(tab, "# FINAL COVERAGE DISTRIBUTION:\n# COVERAGE N_SITES\n");
                for (int c = 0; c < C; c++) fprintf(tab, "# %d %lu\n", c, (unsigned long)fdist[k * (size_t)C + (size_t)c]);
                fprintf(tab, "# FINAL MEAN DEPTH = %lf\n", (double)totcov[k] / processed[k]);
                fprintf(tab, "## Number of sites processed: %lu\n", (unsigned long)processed[k]);
                fprintf(tab, "## Number of sites skipped: %lu\n", (unsigned long)skipped[k]);
                fclose(tab);
            }
            fprintf(sum, "# SEGMENT\tSTART\tEND\tLIBD0\tLIBD1\tLIBD2\tNUM_SITES\n");
            for (int w = 0; w < nw[k]; w++) {
                const size_t i = k * (size_t)maxW + (size_t)w;
                char e0[40], e1[40], e2[40];
                const bool lin = want_linear && wlin[i * 3 + 2] == wlin[i * 3 + 2];
                put_e(e0, lin && !o.ld ? wlin[i * 3] : exp(wll[i * 3]));
                put_e(e1, lin && !o.ld ? wlin[i * 3 + 1] : exp(wll[i * 3 + 1]));
                put_e(e2, lin ? wlin[i * 3 + 2] : exp(wll[i * 3 + 2]));
                fprintf(sum, "%d\t%lu\t%lu\t%s\t%s\t%s\t%d\n", w + 1, (unsigned long)ws[i], (unsigned long)we[i], e0, e1, e2, wn[i]);
            }
            fclose(sum);
            if (o.hiddengem && nw[k] > 0) {  // the table hiddengem prints to stdout (src/hiddengem.c:259-283)
                const std::string hg_fn = o.out_dir + "/" + o.sq_id + "." + smp.name + ".hiddengem.txt";
                FILE *hg = fopen(hg_fn.c_str(), "w");
                if (!hg) {
                    fprintf(stderr, "[::] ERROR: Cannot open '%s' for writing.\n", hg_fn.c_str());
                    return 1;
                }
                fprintf(hg, o.posterior ? "Segment\tIBD0_Score\tIBD1_Score\tIBD2_Score\tInferred_State\tP_IBD0\tP_IBD1\tP_IBD2\n"
                                        : "Segment\tIBD0_Score\tIBD1_Score\tIBD2_Score\tInferred_State\n");
                const int64_t a = hg_off[k], b = hg_off[k + 1];
                char s0[48], s1[48], s2[48];
                for (int64_t i = a; i < b; i++) {
                    put_score_log(s0, hg_score[(size_t)i * 3]);
                    put_score_log(s1, hg_score[(size_t)i * 3 + 1]);
                    put_score_log(s2, hg_score[(size_t)i * 3 + 2]);
                    if (o.posterior)
                        fprintf(hg, "%d\t%s\t%s\t%s\t%d\t%.6f\t%.6f\t%.6f\n", (int)(i - a + 1), s0, s1, s2, (int)hg_state[(size_t)i],
                                hg_post[(size_t)i * 3], hg_post[(size_t)i * 3 + 1], hg_post[(size_t)i * 3 + 2]);
                    else
                        fprintf(hg, "%d\t%s\t%s\t%s\t%d\n", (int)(i - a + 1), s0, s1, s2, (int)hg_state[(size_t)i]);
                }
                const double n = (double)(b - a);
                for (int c = 0; c < 3; c++)
                    fprintf(hg, "#%% IBD%d (n = %.0f): %.2f\n", c, (double)hg_counts[k * 3 + (size_t)c], ((double)hg_counts[k * 3 + (size_t)c] / n) * 100);
                if (o.posterior)
                    for (int c = 0; c < 3; c++)
                        fprintf(hg, "#%% posterior IBD%d (n = %.2f): %.2f\n", c, hg_expected[k * 3 + (size_t)c], (hg_expected[k * 3 + (size_t)c] / n) * 100);
                if (o.share_sd) fputs(share_sd_lines(&hg_expected[k * 3], &hg_cov[k * 9], n).c_str(), hg);
                fclose(hg);
            }
            if (o.tracts && nw[k] > 0) {  // START / END / NUM_SITES from the run's own window bookkeeping
                const std::string tr_fn = o.out_dir + "/" + o.sq_id + "." + smp.name + ".tracts.txt";
                FILE *tf = fopen(tr_fn.c_str(), "w");
                if (!tf) {
                    fprintf(stderr, "[::] ERROR: Cannot open '%s' for writing.\n", tr_fn.c_str());
                    return 1;
                }
                const std::string head = tract_header(false, o.posterior);
                fwrite(head.data(), 1, head.size(), tf);
                const size_t w0 = k * (size_t)maxW;
                for (int64_t j = tr_off[k]; j < tr_off[k + 1]; j++) {
                    const hiddengem_tract &r = tracts[(size_t)j];
                    int64_t sites = 0;
                    for (int64_t w = r.first_bin; w < r.first_bin + r.n_bins; w++) sites += wn[w0 + (size_t)w];
                    const std::string row = tract_row(r, j - tr_off[k], ws[w0 + (size_t)r.first_bin], we[w0 + (size_t)(r.first_bin + r.n_bins - 1)],
                                                      sites, o.posterior);
                    fwrite(row.data(), 1, row.size(), tf);
                }
                fclose(tf);
            }
            return 0;
        };
        const size_t n_writers = std::max<size_t>(1, std::min<size_t>({T, (size_t)WRITER_THREADS, (size_t)std::thread::hardware_concurrency()}));
        std::atomic<size_t> next_k{0};
        std::atomic<int> write_rc{0};
        auto writer = [&] {
            std::vector<char> line(1 << 20);
            for (size_t k; (k = next_k.fetch_add(1)) < T;)
                if (write_target(k, line)) write_rc = 1;
        };
        if (n_writers == 1) {
            writer();
        } else {
            std::vector<std::thread> pool;
            for (size_t i = 0; i < n_writers; i++) pool.emplace_back(writer);
            for (auto &t : pool) t.join();
        }
        if (write_rc) return 1;
    }
    if (psrc && device == 0)
        while (psrc->users.load() > 0) std::this_thread::yield();  // clones may still be copying from this engine's panel
    ibdgem_engine_destroy(e);
    return 0;
}

}  // namespace

int main(int argc, char *argv[]) {
    const clock_t start = clock();
    Options o;
    static int ld_flag = 0, no_tab_flag = 0, hg_flag = 0, post_flag = 0, tracts_flag = 0, share_sd_flag = 0;
    static struct option longopts[] = {{"LD", no_argument, &ld_flag, 1},
                                       {"vcf", required_argument, 0, 'V'},
                                       {"hap", required_argument, 0, 'H'},
                                       {"legend", required_argument, 0, 'L'},
                                       {"indv", required_argument, 0, 'I'},
                                       {"pileup", required_argument, 0, 'P'},
                                       {"pileup-name", required_argument, 0, 'N'},
                                       {"window-size", required_argument, 0, 'w'},
                                       {"allele-freqs", required_argument, 0, 'A'},
                                       {"sample-list", required_argument, 0, 'S'},
                                       {"sample", required_argument, 0, 's'},
                                       {"background-list", required_argument, 0, 'B'},
                                       {"max-cov", required_argument, 0, 'M'},
                                       {"downsample-cov", required_argument, 0, 'D'},
                                       {"out-dir", required_argument, 0, 'O'},
                                       {"max-af", required_argument, 0, 'F'},
                                       {"min-af", required_argument, 0, 'f'},
                                       {"positions", required_argument, 0, 'p'},
                                       {"min-qual", required_argument, 0, 'q'},
                                       {"chromosome", required_argument, 0, 'c'},
                                       {"error-rate", required_argument, 0, 'e'},
                                       {"variable-sites-only", no_argument, 0, 'v'},
                                       {"help", no_argument, 0, 'h'},
                                       {"gpus", required_argument, 0, 1001},     // additive
                                       {"batch", required_argument, 0, 1002},    // additive
                                       {"panel-cache", required_argument, 0, 1003},  // additive
                                       {"no-tab", no_argument, &no_tab_flag, 1},  // additive
                                       {"hiddengem", no_argument, &hg_flag, 1},   // additive: chain the Viterbi pass
                                       {"posterior", no_argument, &post_flag, 1},  // additive: posteriors in the hiddengem files
                                       {"tracts", no_argument, &tracts_flag, 1},   // additive: IBD tracts beside the hiddengem files
                                       {"share-sd", no_argument, &share_sd_flag, 1},  // additive: share sd in the hiddengem files
                                       {"p01", required_argument, 0, 1004},
                                       {"p02", required_argument, 0, 1005},
                                       {"p12", required_argument, 0, 1006},
                                       {0, 0, 0, 0}};
    if (argc == 1) print_help(0);
    char cwd[PATH_MAX];
    o.out_dir = getcwd(cwd, sizeof(cwd)) ? cwd : "./";
    int option;
    while ((option = getopt_long(argc, argv, ":V:H:L:I:P:w:N:A:S:s:B:p:q:M:F:f:D:O:c:e:vh", longopts, nullptr)) != -1) {
        switch (option) {
            case 0: break;
            case 'V': o.in_vcf = 1; o.vcf_fn = optarg; break;
            case 'H': o.in_impute = 1; o.hap_fn = optarg; break;
            case 'L': o.in_impute = 1; o.legend_fn = optarg; break;
            case 'I': o.in_impute = 1; o.indv_fn = optarg; break;
            case 'P': o.pu_fn = optarg; break;
            case 'w': o.window = atoi(optarg); break;
            case 'N': o.sq_id = optarg; break;
            case 'S': o.opt_s1 = 1; o.sample_fn = optarg; break;
            case 's': o.opt_s2 = 1; o.sample_str = optarg; break;
            case 'B': o.opt_b = 1; o.ref_fn = optarg; break;
            case 'A': o.opt_a = 1; o.af_fn = optarg; break;
            case 'M': o.max_cov = (unsigned)atoi(optarg); break;
            case 'F': o.max_af = atof(optarg); break;
            case 'f': o.min_af = atof(optarg); break;
            case 'p': o.opt_p = 1; o.pos_fn = optarg; break;
            case 'q': o.min_qual = atof(optarg); break;
            case 'c': o.uchr = optarg; break;
            case 'e': o.epsilon = atof(optarg); break;
            case 'O': o.out_dir = optarg; break;
            case 'D': o.target_dp = atof(optarg); o.opt_d = 1; break;
            case 'v': o.opt_v = 1; break;
            case 'h': print_help(0); break;
            case 1001: o.gpus = atoi(optarg); break;
            case 1002: o.batch = atoi(optarg); break;
            case 1003: o.cache_fn = optarg; break;
            case 1004: o.p01 = atof(optarg); break;
            case 1005: o.p02 = atof(optarg); break;
            case 1006: o.p12 = atof(optarg); break;
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
    o.ld = ld_flag;
    o.no_tab = no_tab_flag;
    o.hiddengem = hg_flag;
    o.posterior = post_flag;
    o.tracts = tracts_flag;
    o.share_sd = share_sd_flag;
    for (int i = optind; i < argc; i++) fprintf(stderr, "Given extra argument %s.\n", argv[i]);
    // validation: the reference exits with status 0 on invalid values (src/ibdgem.c:966-989)
    if (o.opt_d && o.target_dp <= 0) {
        fprintf(stderr, "[::] ERROR: Invalid down-sample coverage (-D) of %.2f (must be > 0).\n", o.target_dp);
        exit(0);
    }
    if (o.min_af < 0) {
        fprintf(stderr, "[::] ERROR: Invalid minimum alternate allele frequency (-f) of %.2f (must be >= 0).\n", o.min_af);
        exit(0);
    }
    if (o.max_af > 1) {
        fprintf(stderr, "[::] ERROR: Invalid maximum alternate allele frequency (-F) of %.2f (must be <= 1).\n", o.max_af);
        exit(0);
    }
    if (o.max_cov < 1) {
        fprintf(stderr, "[::] ERROR: Invalid maximum estimated coverage (-M) of %u (must be >= 1).\n", o.max_cov);
        exit(0);
    }
    if (o.min_qual < 0) {
        fprintf(stderr, "[::] ERROR: Invalid genotype quality minimum (-q) of %.2f (must be >= 0).\n", o.min_qual);
        exit(0);
    }
    if (o.window < 2) {
        fprintf(stderr, "[::] ERROR: Invalid window size (-w) of %d (must be >= 2).\n", o.window);
        exit(0);
    }
    if (o.posterior && !o.hiddengem) {
        fprintf(stderr, "[::] ERROR: --posterior needs --hiddengem (the posteriors are written to the hiddengem files).\n");
        exit(0);
    }
    if (o.share_sd && !o.posterior) {
        fprintf(stderr, "[::] ERROR: --share-sd needs --posterior (the standard deviations are those of the posterior counts).\n");
        exit(0);
    }
    if (o.tracts && !o.hiddengem) {
        fprintf(stderr, "[::] ERROR: --tracts needs --hiddengem (the tracts are runs of the hiddengem states).\n");
        exit(0);
    }
    if (o.max_cov > IBDGEM_MAX_COV_LIMIT) o.max_cov = IBDGEM_MAX_COV_LIMIT;  // pileup lines with cov >= 128 never load

    Shared sh;
    sh.opt = &o;
    sh.user_cmd = argv[0];
    sh.user_cmd += " ";
    for (int i = 1; i < argc; i++) {
        sh.user_cmd += argv[i];
        sh.user_cmd += " ";
    }

    PileupStore pu;
    if (load_pileup(o.pu_fn, o.uchr, &pu)) {
        fprintf(stderr, "[::] ERROR parsing Pileup data; make sure input is valid.\n");
        exit(1);
    }
    FreqTable af;
    std::unordered_set<uint64_t> positions;
    PackOptions po;
    po.min_qual = o.min_qual;
    if (o.opt_a) {
        if (read_af(o.af_fn, o.uchr, &af)) exit(1);
        po.af = &af;
    }
    if (o.opt_p) {
        if (read_positions(o.pos_fn, o.uchr, &positions)) exit(1);
        po.positions = &positions;
    }
    if (!o.in_vcf && !o.in_impute) {
        fprintf(stderr, "[::] ERROR: Missing genotype files.\n");
        exit(1);
    }
    if (o.in_vcf && o.in_impute) {
        fprintf(stderr, "[::] ERROR: 2 types of genotype inputs detected. Please choose either IMPUTE or VCF format.\n");
        exit(1);
    }
    PackedPanel panel;
    if (o.in_vcf) {
        if (!o.cache_fn.empty()) {
            bool hit = false;
            if (pack_vcf_cached(o.vcf_fn, o.cache_fn, pu, po, &panel, &hit)) exit(1);
            fprintf(stderr, "[::] panel cache %s: %s\n", o.cache_fn.c_str(), hit ? "loaded" : "written");
        } else if (pack_vcf(o.vcf_fn, pu, po, &panel)) {
            exit(1);
        }
    } else {
        std::vector<std::string> names;
        {
            FILE *fh = fopen(o.hap_fn.c_str(), "r"), *fl = fopen(o.legend_fn.c_str(), "r");
            const bool ok = fh && fl;
            if (fh) fclose(fh);
            if (fl) fclose(fl);
            if (!ok) {
                fprintf(stderr, "[::] ERROR parsing hap/legend/indv data; make sure inputs are valid.\n");
                exit(1);
            }
        }
        if (!o.cache_fn.empty()) {
            // binary cache of the parsed panel: later runs against the same panel (other pileups, other
            // options) skip the text files
            bool hit = false;
            if (pack_impute_cached(o.hap_fn, o.legend_fn, o.indv_fn, o.cache_fn, pu, po, &panel, &hit)) exit(1);
            fprintf(stderr, "[::] panel cache %s: %s\n", o.cache_fn.c_str(), hit ? "loaded" : "written");
        } else {
            if (read_indv(o.indv_fn, &names)) exit(1);
            if (pack_impute(o.hap_fn, o.legend_fn, names, pu, po, &panel)) exit(1);
        }
    }
    if (o.opt_s1) {
        if (read_sample_file(o.sample_fn, panel.names, false, &sh.targets)) exit(1);
    } else if (o.opt_s2) {
        if (read_sample_string(o.sample_str, panel.names, &sh.targets)) exit(1);
    } else {
        for (size_t i = 0; i < panel.names.size(); i++) sh.targets.push_back({panel.names[i], (int32_t)i});
    }
    if (o.opt_b) {
        if (read_sample_file(o.ref_fn, panel.names, true, &sh.background)) exit(1);
    } else {
        for (size_t i = 0; i < panel.names.size(); i++) sh.background.push_back({panel.names[i], (int32_t)i});
    }
    sh.pu_idx = find_sample(panel.names, o.sq_id);
    const InputDist dist = input_distribution(pu, o);
    sh.panel = &panel;
    sh.pu = &pu;
    sh.dist = &dist;
    if (panel.S == 0) {
        fprintf(stderr, "[::] ERROR: the genotype panel has no site lines.\n");
        exit(1);
    }

    if (dist.cull_p != 1.0) {
        // -D thinning (cull_dp, src/ibdgem.c:126-137, 627-628): glibc rand() from its default seed,
        // consumed target by target, site by site, REF bases then ALT bases, only at sites that pass
        // every filter for that target.  The filter verdicts come from the engine's site table.
        ibdgem_params prm{};
        prm.epsilon = o.epsilon; prm.max_cov = o.max_cov; prm.window_size = o.window;
        prm.min_af = o.min_af; prm.max_af = o.max_af; prm.variable_sites_only = o.opt_v; prm.device = 0;
        ibdgem_engine *e = nullptr;
        const size_t S = (size_t)panel.S;
        std::vector<uint8_t> st(S);
        if (ibdgem_engine_create(&prm, &e) ||
            ibdgem_engine_upload_sites(e, panel.S, panel.pos.data(), panel.n_ref.data(), panel.n_alt.data(), panel.host_keep.data(),
                                       panel.af_user.empty() ? nullptr : panel.af_user.data()) ||
            ibdgem_engine_upload_panel(e, panel.S, panel.N, panel.bits.data(), panel.Wh) ||
            ibdgem_engine_get_site_table(e, nullptr, st.data(), nullptr)) {
            fprintf(stderr, "%s\n", ibdgem_last_error());
            exit(1);
        }
        ibdgem_engine_destroy(e);
        sh.tgt_counts.assign(sh.targets.size() * S * 2, 0);
        for (size_t k = 0; k < sh.targets.size(); k++) {
            const size_t h0 = 2 * (size_t)sh.targets[k].ordinal;
            for (size_t s = 0; s < S; s++) {
                if (!st[s]) continue;
                if (o.opt_v) {
                    const uint32_t *row = panel.bits.data() + s * (size_t)panel.Wh;
                    if (!((row[h0 >> 5] >> (h0 & 31)) & 1u) && !((row[(h0 + 1) >> 5] >> ((h0 + 1) & 31)) & 1u)) continue;
                }
                for (int j = 0; j < 2; j++) {
                    const unsigned c = j ? panel.n_alt[s] : panel.n_ref[s];
                    unsigned kept = 0;
                    for (unsigned i = 0; i < c; i++)
                        if ((rand() / (double)RAND_MAX) < dist.cull_p) kept++;
                    sh.tgt_counts[(k * S + s) * 2 + (size_t)j] = (uint8_t)kept;
                }
            }
        }
    }

    const int gpus = std::max(1, std::min<int>(o.gpus, (int)sh.targets.size()));
    int rc = 0;
    if (gpus == 1) {
        rc = run_shard(&sh, 0, 0, sh.targets.size());
    } else {  // contiguous shards of the target list, one host thread and one engine per device
        std::vector<std::thread> th;
        std::vector<int> rcs((size_t)gpus, 0);
        const size_t n = sh.targets.size();
        PanelSource psrc;
        psrc.users = gpus - 1;
        for (int d = 0; d < gpus; d++) {
            const size_t base = n / (size_t)gpus, extra = n % (size_t)gpus;
            const size_t lo = (size_t)d * base + std::min<size_t>((size_t)d, extra), hi = lo + base + ((size_t)d < extra ? 1 : 0);
            th.emplace_back([&, d, lo, hi] { rcs[(size_t)d] = run_shard(&sh, d, lo, hi, &psrc); });
        }
        for (auto &t : th) t.join();
        for (int r : rcs) rc |= r;
    }
    if (rc) exit(1);
    const double minutes = ((double)(clock() - start) / CLOCKS_PER_SEC) / 60;
    fprintf(stderr, "Run time: %f minutes.\n", minutes);
    return EXIT_SUCCESS;
}
