/* ibdgem_b200.h — C ABI of the B200-native IBDGem likelihood engine (libibdgem_b200.so).
 *
 * This is the drop-in boundary for the scoring path of Paleogenomics/IBDGem.  The reference has
 * no plugin/FFI interface (SURVEY.md §8b); its only library-like seam is src/ibd-math.h:14-63 and
 * the arithmetic open-coded in compare_impute / compare_vcf (src/ibdgem.c:185-476, 498-775) and
 * hiddengem's calc_score (src/hiddengem.c:108-147).  Each entry point below names the reference
 * code it replaces.  Conventions follow the reference (SURVEY.md §8b "Ownership"/"Errors"):
 *   - plain pointers and sizes only; the caller owns every host buffer; the engine owns device
 *     copies; nothing is retained after a call returns except what upload_* copied to HBM;
 *   - every function returns int, 0 = ok, non-zero = error with a message available from
 *     ibdgem_last_error() (prefixed "[::] ERROR" like the reference's stderr messages);
 *   - one engine per process x device; calls on one engine are serialised by the caller;
 *   - there is NO CPU fallback: without a usable CUDA device create() fails.
 *
 * Haplotype convention (src/ibd-parse.c:29, src/ibdgem.c:638-639): individual ordinal i owns
 * haplotypes 2i and 2i+1 — the characters at offsets 4i and 4i+2 of a .hap line.
 */
#ifndef IBDGEM_B200_H
#define IBDGEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IBDGEM_B200_ABI_VERSION 2
#define IBDGEM_MAX_COV_LIMIT 127 /* src/pileup.h:12 MAX_COV 128: lines with cov >= 128 are dropped */

typedef struct ibdgem_engine ibdgem_engine;

/* The file-scope option statics of src/ibdgem.c:21-38 that the arithmetic reads. */
typedef struct ibdgem_params {
    double epsilon;               /* -e  EPSILON        default 0.02 */
    uint32_t max_cov;             /* -M  USER_MAX_COV   default 20, 1..127 */
    int32_t window_size;          /* -w  WINDOWSIZE     default 100, >= 2 */
    double min_af;                /* -f  USER_MIN_AF    default 0 */
    double max_af;                /* -F  USER_MAX_AF    default 1 */
    int32_t variable_sites_only;  /* -v  OPT_V */
    int32_t device;               /* CUDA device ordinal */
} ibdgem_params;

/* Site status codes written by the engine. */
enum {
    IBDGEM_SITE_SKIPPED = 0,     /* counted in "sites skipped" (src/ibdgem.c:584-626) */
    IBDGEM_SITE_INFORMATIVE = 1, /* processed, advances the window (src/ibdgem.c:665-733) */
    IBDGEM_SITE_ZERO_DATA = 2    /* processed, printed with likelihoods 1.0, not aggregated (:657-663) */
};

/* Per-call outputs.  Every pointer is a caller-allocated HOST buffer and may be NULL to skip
 * that output.  T = n_targets of the call, S = uploaded sites, C = max_cov + 1. */
typedef struct ibdgem_scores {
    int32_t max_windows;       /* capacity of the per-window arrays, per target */
    int32_t *n_windows;        /* [T]        number of windows emitted (src/ibdgem.c:736-759) */
    uint64_t *w_start;         /* [T][maxW]  sgmt_start — position of the first kept site */
    uint64_t *w_end;           /* [T][maxW]  sgmt_end   — position of the last kept site */
    int32_t *w_nsites;         /* [T][maxW]  snp_count */
    double *w_loglik;          /* [T][maxW][3] natural log of LIBD0, LIBD1, LIBD2 of the summary row */
    uint64_t *processed;       /* [T] "## Number of sites processed" */
    uint64_t *skipped;         /* [T] "## Number of sites skipped" */
    uint64_t *final_total_cov; /* [T] numerator of "# FINAL MEAN DEPTH" (src/ibdgem.c:629,766) */
    uint64_t *final_dist;      /* [T][C] "# FINAL COVERAGE DISTRIBUTION" */
    uint8_t *site_status;      /* [T][S]    optional expanded per-target site status */
    double *site_lik;          /* [T][S][3] optional expanded LIBD0, LIBD1, LIBD2 of each tab row (linear) */
    double *w_lik_linear;      /* [T][maxW][3] optional: the reference's OWN window aggregates — running fp64 products of
                                  the per-site likelihoods in file order, starting from 1.0 (sum_ibd0 *= ibd0 ...,
                                  src/ibdgem.c:562, 665-667) — bit for bit, underflow to denormals and 0 included, so
                                  that a formatter can print summary.txt columns identical to the reference's.  These are
                                  the three columns of a non-LD row and the LIBD2 column of an --LD row (the --LD means
                                  over the background have no linear-space twin; take those from w_loglik).  Not
                                  available for --LD runs with -v / -D (rows stay NaN). */
    void *w_loglik_device;     /* optional DEVICE pointer: [T][maxW][3] doubles are also written here, for the
                                  device-resident hiddengem front-end or as this rank's block of a gathered
                                  table in another GPU's memory (ibdgem_peer_open).  The tensor --LD path
                                  writes columns [0, n_windows) of every row, range by range; the other
                                  paths write whole rows (columns past n_windows are NaN). */
} ibdgem_scores;

/* ---- lifetime --------------------------------------------------------------------------- */

/* Replaces init_nCk + the per-site find_pDgG calls (src/ibd-math.c:13-81, src/ibdgem.c:632-634,
 * 1168): builds the P(D|G) table for every (n_ref, n_alt) class on the host with libm pow(), in
 * the reference's evaluation order, and uploads it. */
int ibdgem_engine_create(const ibdgem_params *params, ibdgem_engine **out);
int ibdgem_engine_destroy(ibdgem_engine *e); /* NULL tolerated, like destroy_nCk (src/ibd-math.c:34-43) */
const char *ibdgem_last_error(void);
int ibdgem_abi_version(void);

/* All engine work is enqueued on this CUDA stream (a cudaStream_t passed as void*; NULL = the
 * legacy default stream).  Lets a caller time the engine with its own events. */
int ibdgem_engine_set_stream(ibdgem_engine *e, void *cuda_stream);

/* ---- inputs (host packer -> HBM) --------------------------------------------------------- */

/* Per panel line i (one .hap/.legend line or one VCF record), what the host-side parsers
 * produced (src/ibdgem.c:589-608, 621-622; src/pileup.c:442-485):
 *   pos[i]       legend/VCF position
 *   n_ref[i]     pileup bases equal to REF, n_alt[i] pileup bases equal to ALT (before -D)
 *   host_keep[i] 1 iff the line parsed, is a SNP, has a pileup line and passes -p (and, for VCF,
 *                the biallelic/GT/QUAL checks) — every filter that does not need the panel row
 *   af_user[i]   NaN, or the -A allele frequency found for pos[i]; the whole array may be NULL */
int ibdgem_engine_upload_sites(ibdgem_engine *e, int64_t n_sites, const uint64_t *pos,
                               const uint8_t *n_ref, const uint8_t *n_alt, const uint8_t *host_keep,
                               const double *af_user);

/* Bit-packed phased panel, site-major: row i holds the 2*n_indiv alleles of panel line i,
 * haplotype h in bit (h & 31) of word (h >> 5); words_per_site >= ceil(2*n_indiv/32), padding
 * bits zero.  Replaces the per-target re-read of the .hap file (src/ibdgem.c:573, 771). */
int ibdgem_engine_upload_panel(ibdgem_engine *e, int64_t n_sites, int32_t n_indiv,
                               const uint32_t *bits, int64_t words_per_site);
/* The panel copy is issued in site chunks on the engine's copy stream and may still be in flight
 * when upload_panel returns: `bits` must stay valid and unchanged until the next call on this engine
 * that returns results (prepare / get_site_table / score_* all wait for what they read), or until
 * ibdgem_engine_sync_uploads().  With page-locked `bits` the copy overlaps the scoring of the windows
 * whose rows have already arrived; with pageable memory it is simply complete on return. */
int ibdgem_engine_sync_uploads(ibdgem_engine *e);

/* Panel already in device memory.  Multi-GPU use: the packed panel is identical on every rank, so each
 * rank copies 1/N of it over PCIe and the ranks exchange the pieces over NVLink (one all_gather per
 * piece; ibdgem_b200/shard.py replicate_panel) instead of N full uploads through the host bridges.
 * `d_bits` is caller-owned device memory in the layout of ibdgem_engine_upload_panel; it must stay
 * valid and, once declared ready, unchanged until another panel is set or the engine is destroyed.
 * Rows become readable in pieces: after set_panel_device none is; every
 * ibdgem_engine_panel_rows_ready(e, row_end, stream) declares rows [0, row_end) complete once the work
 * enqueued so far on `stream` (a cudaStream_t passed as void*; NULL = the engine's own stream) has run.
 * row_end must not decrease; scoring proceeds window range by window range as the pieces are declared,
 * exactly as with upload_panel's own chunks, and fails if it needs rows that were never declared. */
int ibdgem_engine_set_panel_device(ibdgem_engine *e, int64_t n_sites, int32_t n_indiv,
                                   const uint32_t *d_bits, int64_t words_per_site);
int ibdgem_engine_panel_rows_ready(ibdgem_engine *e, int64_t row_end, void *stream);

/* Panel copied from another engine of the same process (usually on another GPU), device to device over NVLink, chunk
 * by chunk as the source's own upload lands: `ibdgem --gpus N` uploads the panel over PCIe once and clones it N-1
 * times.  `src` must stay alive, with its panel unchanged, until this engine's next call that returns results. */
int ibdgem_engine_clone_panel(ibdgem_engine *e, ibdgem_engine *src);

/* Target-independent stage: allele frequency by popcount over the packed row (find_f_impute /
 * find_f_vcf, src/ibd-parse.c:91-110), the AF-range and max-cov filters (src/ibdgem.c:616-626),
 * per-site IBD0 / IBD1[g] / IBD2[g] (find_pDgf, find_pDgIBD1, src/ibd-math.c:84-142) and the
 * shared window map.  Called implicitly by the score functions when inputs changed. */
int ibdgem_engine_prepare(ibdgem_engine *e);
/* Marks the prepared state stale without touching the uploaded inputs, so the next prepare() /
 * score_*() recomputes the whole target-independent stage from the packed arrays resident in
 * HBM (what one reference run does per invocation).  Device buffers are kept. */
int ibdgem_engine_invalidate(ibdgem_engine *e);

/* Compact per-site table after prepare() (any pointer may be NULL):
 *   f[S]; status[S] (for a target that is not filtered by -v/-D);
 *   lik7[S][7] = { IBD0, IBD1|g=0, IBD1|g=1, IBD1|g=2, P(D|00), P(D|01), P(D|11) } — the tab.txt
 *   likelihood columns of target t at site i are lik7[i][0], lik7[i][1+g], lik7[i][4+g]. */
int ibdgem_engine_get_site_table(ibdgem_engine *e, double *f, uint8_t *status, double *lik7);

/* ---- multi-GPU ---------------------------------------------------------------------------- */

/* Two partitions of a run across the GPUs of a node (SURVEY.md 8e; both follow from the independence of
 * targets, src/ibdgem.c:522, and of windows, :558-578):
 *   - by TARGETS: every rank scores its own slice of the target list (any mode).  Nothing to set here:
 *     pass the slice to score_*.
 *   - by WINDOWS (shared window maps only: --LD on the tensor path, no -v / -D): rank `index` of `count`
 *     scores windows [nW*index/count, nW*(index+1)/count) of EVERY target.  Everything a rank does then
 *     scales with 1/count — including the panel rows it needs: only rows [site_begin, site_end) reported
 *     by ibdgem_engine_window_shard() are read, so a rank may place just those rows in a device buffer
 *     handed over with ibdgem_engine_set_panel_device (the rest of the buffer is never touched).
 *     Score calls write only the shard's columns of w_loglik / w_loglik_device; the bookkeeping arrays
 *     and n_windows describe all windows on every rank. */
int ibdgem_engine_set_window_shard(ibdgem_engine *e, int32_t index, int32_t count);
int ibdgem_engine_window_shard(ibdgem_engine *e, int32_t *w_begin, int32_t *w_end, int64_t *site_begin,
                               int64_t *site_end); /* prepares the window map if necessary */
/* With a window shard set, have score_ld write the HOST table ibdgem_scores.w_loglik compactly and WINDOW-major, as
 * [w_end - w_begin][T][3] (only the shard's windows exist): contiguous device-to-host copies, issued sub-range by
 * sub-range under the scoring of the next one, instead of T short strided rows (10,000 rows of 3 KB at C5 over
 * 8 GPUs).  The device table w_loglik_device keeps the full [T][max_windows][3] layout. */
int ibdgem_engine_set_shard_compact_output(ibdgem_engine *e, int32_t on);

/* Gather of per-window scores over NVLink without a rendezvous inside the scoring loop: the root
 * allocates the gathered table with ibdgem_peer_alloc (cudaMalloc + a 64-byte CUDA IPC handle), the other
 * ranks of the node map it with ibdgem_peer_open, and every rank passes its own block (or, for window
 * shards, the table itself) as ibdgem_scores.w_loglik_device: the engine then stores each finished window
 * range straight into the root's memory while later ranges are still being scored.  The handle travels
 * between processes by any means (the Python mirror broadcasts it with torch.distributed). */
int ibdgem_peer_alloc(int32_t device, int64_t bytes, void **dptr, unsigned char *handle64);
int ibdgem_peer_open(int32_t device, const unsigned char *handle64, void **dptr);
int ibdgem_peer_close(int32_t device, void *dptr, int32_t owner);

/* ---- scoring ----------------------------------------------------------------------------- */

/* Non-LD comparison of the pileup against each target: the per-target body of compare_impute /
 * compare_vcf without the --LD block (src/ibdgem.c:550-668, 723-768).
 *   targets[T]       individual ordinals, in output order
 *   tgt_counts       NULL, or [T][S][2] down-sampled (n_ref, n_alt) per target (-D,
 *                    src/ibdgem.c:627-628; the host draws them with rand() in reference order) */
int ibdgem_engine_score_nonld(ibdgem_engine *e, int32_t n_targets, const int32_t *targets,
                              const uint8_t *tgt_counts, ibdgem_scores *out);

/* --LD comparison (src/ibdgem.c:669-722, 737-753): LIBD0 = mean over background individuals of
 * the window product of P(D|G_bg); LIBD1 = mean over background x 4 haplotype pairings; LIBD2 as
 * in non-LD.  bg[n_bg] are background ordinals (refids, duplicates allowed); members equal to
 * the target or to pu_idx (-N naming a panel member, or -1) are excluded and the divisor
 * shrinks accordingly (src/ibdgem.c:714, 742-749). */
int ibdgem_engine_score_ld(ibdgem_engine *e, int32_t n_targets, const int32_t *targets,
                           int32_t n_bg, const int32_t *bg, int32_t pu_idx,
                           const uint8_t *tgt_counts, ibdgem_scores *out);

/* Which --LD implementation the last score_ld call used:
 *   1 = tensor-core window GEMM with fused log-sum-exp (shared windows: no -v, no -D; ld_mma.cu),
 *   2 = tensor-core GEMM over per-target windows (-v, -D; rows are (target, window) pairs; ld_vmma.cu),
 *   0 = general CUDA-core path (class tables that are not depth-linear, windows above 1,024 sites without -v/-D,
 *       forced). */
int ibdgem_engine_last_ld_path(ibdgem_engine *e);
/* Force the general path (testing / A-B measurement). */
int ibdgem_engine_force_general_ld(ibdgem_engine *e, int on);

/* ---- hiddengem --------------------------------------------------------------------------- */

/* Batched three-state Viterbi (init_summary + calc_score + backtrace, src/hiddengem.c:51-147,
 * 246-283) over n_tables independent summary tables.
 *   lik            [sum(n_bins)][3] per-bin LIBD0/1/2 as parsed from summary files
 *                  (is_log = 0), or their natural logs straight from the engine (is_log = 1)
 *   bin_offsets    [n_tables + 1] prefix offsets of each table's bins
 *   state          [sum(n_bins)]  Inferred_State
 *   score_log      [sum(n_bins)][3] natural log of the reference's running-product scores
 *   state_counts   [n_tables][3]  bins per state (the "#% IBDk" lines) */
int hiddengem_viterbi_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets,
                            const double *lik, int32_t is_log, double p01, double p02, double p12,
                            uint8_t *state, double *score_log, int64_t *state_counts);

/* The same on DEVICE buffers (SURVEY.md 8f-3: window scores that never left the GPU are not re-parsed from 7-digit
 * text, src/hiddengem.c:66-76).  d_lik / d_state / d_score_log / d_state_counts are device pointers on the engine's
 * GPU; bin_offsets is a HOST array of n_tables + 1 prefix offsets.
 *   table_stride = 0   tables are packed: table t holds bins [bin_offsets[t], bin_offsets[t+1]) of every array;
 *   table_stride > 0   table t starts at bin t * table_stride and has bin_offsets[t+1] - bin_offsets[t] bins — with
 *                      table_stride = max_windows and is_log = 1 this consumes ibdgem_scores.w_loglik_device as is. */
int hiddengem_viterbi_batch_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                   const double *d_lik, int32_t is_log, double p01, double p02, double p12,
                                   uint8_t *d_state, double *d_score_log, int64_t *d_state_counts);
/* Near-tie guard: the recursion runs on sums of fp64 logarithms where the reference multiplies x87 long doubles
 * (src/hiddengem.c:43, 110-141).  A table in which some arg-max is decided by less than the rounding error those sums
 * can have accumulated — or, on the text path, whose scores leave the range of a normal long double — is re-evaluated
 * on the host with the reference's own long double recurrence.  Returns how many tables of the last call were. */
int64_t hiddengem_last_flagged(ibdgem_engine *e);

/* Posterior IBD-state probabilities of every bin, by forward-backward over the SAME path weights the Viterbi entries
 * maximise (src/hiddengem.c:108-147): for one table of n bins and a state path x,
 *     W(x) = prod_{i<n} nrm[i][x_i] * prod_{0<i<n} pen(x_{i-1}, x_i),    posterior[i][s] = sum_{x: x_i = s} W(x) / sum_x W(x)
 * with pen = 1 on the diagonal and p01 / p02 / p12 off it (symmetric), no prior on bin 0, and nrm the per-bin
 * normalisation hiddengem applies: l_s / ((l0 + l1) + l2) for is_log = 0, exp(L_s - m) / sum_k exp(L_k - m) with m the
 * row maximum for is_log = 1.  The penalties are weights, not transition probabilities: this is the marginal of the
 * weights hiddengem already uses, and the Viterbi path is its mode.
 *   - A bin whose normalised row is undefined (all three likelihoods 0 or a NaN total; a NaN score, or a row maximum
 *     that is not finite) gets the uniform emission (1, 1, 1): it carries no information.  (The Viterbi entries
 *     propagate such a bin as the reference does.)
 *   - Penalties may be any finite value >= 0, above 1 included; anything else is an error.  A table whose total
 *     weight is 0 as a real number (possible only with zero penalties) gets NaN posteriors and NaN expected counts;
 *     every other table gets the posteriors of the formula above, however far apart its states are.  Penalties with
 *     max(1, p) / min(1, p) <= 2^400 (no zero among them) run in scaled fp64 linear space, all others in natural-log
 *     arithmetic, which is slower but has no range limit.
 *   - An empty table has no posterior rows and expected counts 0; one bin has posterior = nrm.
 *   lik / bin_offsets   as for the Viterbi entry (host arrays)
 *   posterior           [sum(n_bins)][3], rows sum to 1
 *   expected            [n_tables][3] expected bins per state, sum over the table's bins of posterior */
int hiddengem_posterior_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik,
                              int32_t is_log, double p01, double p02, double p12,
                              double *posterior, double *expected);
/* The same on DEVICE buffers of the engine's GPU (bin_offsets stays a HOST array), with the layouts of the Viterbi
 * device entry: table_stride = 0 for packed tables; table_stride > 0 for table t at bin t * table_stride, which with
 * table_stride = max_windows and is_log = 1 consumes ibdgem_scores.w_loglik_device as is.  Posteriors are written at
 * the positions of the inputs; nothing past a table's bins is written. */
int hiddengem_posterior_batch_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                     const double *d_lik, int32_t is_log, double p01, double p02, double p12,
                                     double *d_posterior, double *d_expected);

/* Posterior moments: the posterior entries' model, emissions, uniform rule and penalties, plus the 3 x 3 posterior
 * covariance of N_s = #{i : x_i = s}, the bins a path puts in state s.  expected[t][s] = E[N_s] (the posterior
 * entries' expected, bit for bit, as are the posteriors) and cov[t][s][u] = Cov(N_s, N_u), exact in the model: one
 * extra recursion in the backward pass, h_i^u[k] = E[#{j > i : x_j = u} | x_i = k], and
 *     Cov(N_s, N_u) = sum_i gamma_i(s) (delta_su - gamma_i(u)) + gamma_i(s) (h_i^u[s] - H_i^u) + gamma_i(u) (h_i^s[u] - H_i^s)
 * with gamma the posteriors and H_i^u = sum_k gamma_i(k) h_i^u[k] (the centred form: no E[N_s N_u] - E[N_s] E[N_u]).
 * Each table's sums run over its bins in a fixed order: the same inputs give the same bits in any batch or layout.
 * Rows of cov sum to 0 (sum_s N_s = n) and cov is positive semi-definite, both up to rounding.
 *   - An empty table has expected 0 and cov 0; one bin has cov = diag(gamma) - gamma gamma^T; a table of total
 *     weight 0 has NaN expected and NaN cov.
 *   - Independent tables (e.g. the chromosomes of one pair) add: the means and covariances of the genome are the sums
 *     of the tables'.  The sd of the IBD1 share is sqrt(cov[1][1]) / n; the kinship phi = (N_1 / 4 + N_2 / 2) / n has
 *     variance (cov[1][1] / 16 + cov[2][2] / 4 + cov[1][2] / 4) / n^2.
 *   posterior   [sum(n_bins)][3] or NULL: with NULL no per-bin array is written, and only 96 B per table come back
 *   expected    [n_tables][3]
 *   cov         [n_tables][3][3], symmetric
 * Arguments, penalties and bin_offsets are checked as by hiddengem_posterior_batch. */
int hiddengem_posterior_moments_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik,
                                      int32_t is_log, double p01, double p02, double p12,
                                      double *posterior, double *expected, double *cov);
/* The same on DEVICE buffers (bin_offsets a HOST array), with the layouts of hiddengem_posterior_batch_device
 * (table_stride = max_windows takes ibdgem_scores.w_loglik_device as is); d_posterior may be NULL. */
int hiddengem_posterior_moments_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                       const double *d_lik, int32_t is_log, double p01, double p02, double p12,
                                       double *d_posterior, double *d_expected, double *d_cov);

/* IBD tracts.  A tract is a maximal run [first_bin, first_bin + n_bins) of bins of one table with the same Viterbi
 * state (in IBDGem a "segment" is one window, i.e. one bin).  Tracts never cross tables; an empty table has none.
 * Records are ordered table by table, then by first_bin; table t's are records [tract_offsets[t], tract_offsets[t+1]).
 *   loglik[s]    sum over the tract's bins of the natural log of the RAW likelihood of state s: the input as is for
 *                is_log = 1, ln l_s for is_log = 0 (a zero likelihood gives -inf, a NaN row NaN sums).  Differences
 *                between states are the tract's log likelihood ratios; the called state need not have the largest,
 *                since penalties can outweigh it.
 *   post_mean    mean over the tract's bins of the posterior of `state`, and post_min its minimum; both NaN without
 *   post_min     posteriors, or when any of them is NaN (a table of zero total weight).
 * Sums are reduced in a fixed order: the same inputs give the same bits. */
typedef struct {            /* 64 bytes, layout fixed */
    int64_t first_bin;      /* 0-based within its table */
    int64_t n_bins;
    int32_t state;          /* 0, 1, 2 = IBD0/1/2 */
    int32_t reserved;       /* 0 */
    double  loglik[3];      /* sum of ln likelihood of each state over the tract */
    double  post_mean;      /* mean posterior of `state` over the tract; NaN without posteriors */
    double  post_min;
} hiddengem_tract;

/* Viterbi (with its near-tie guard: the states are exactly those of hiddengem_viterbi_batch, and
 * hiddengem_last_flagged reports the call's flagged tables) + optional posterior (with_posterior != 0; penalties
 * checked as by hiddengem_posterior_batch) + tracts on the GPU; per-bin arrays never leave the device.  lik /
 * bin_offsets / is_log as for hiddengem_viterbi_batch (host arrays).  tract_offsets: host [n_tables + 1]; the records
 * stay in the engine for hiddengem_last_tracts. */
int hiddengem_tracts_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik, int32_t is_log,
                           double p01, double p02, double p12, int32_t with_posterior, int64_t *tract_offsets);
/* Tracts of states (and posteriors; d_posterior may be NULL) already on the device, e.g. from the two *_device
 * entries, with their layouts (table_stride = 0 packed, > 0 table t at bin t * table_stride).  d_lik is the input those
 * entries took.  A state byte above 2 fails the call. */
int hiddengem_tracts_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                            const double *d_lik, int32_t is_log, const uint8_t *d_state, const double *d_posterior,
                            int64_t *tract_offsets);
/* Copy the records of the last successful tract call (tract_offsets[n_tables] of them) to dst, host memory or
 * (dst_on_device != 0) device memory of the engine's GPU.  Fails if no tract call has succeeded on this engine. */
int hiddengem_last_tracts(ibdgem_engine *e, hiddengem_tract *dst, int32_t dst_on_device);

/* ---- instrumentation --------------------------------------------------------------------- */

/* When enabled every kernel launch is bracketed by CUDA events on the engine stream. */
int ibdgem_engine_enable_timing(ibdgem_engine *e, int on);
int ibdgem_engine_reset_stats(ibdgem_engine *e);
int ibdgem_engine_num_kernels(ibdgem_engine *e);
/* name_out (capacity name_cap), accumulated device milliseconds and launch count of kernel k. */
int ibdgem_engine_kernel_stats(ibdgem_engine *e, int32_t k, char *name_out, int32_t name_cap,
                               double *ms_total, int64_t *launches);
/* Bytes resident in HBM for this engine. */
int64_t ibdgem_engine_device_bytes(ibdgem_engine *e);

#ifdef __cplusplus
}
#endif
#endif /* IBDGEM_B200_H */
