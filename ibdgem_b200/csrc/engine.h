// engine.h — internal declarations shared by the translation units of libibdgem_b200.so.
// Nothing here is part of the ABI (that is include/ibdgem_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <string>
#include <vector>

#include "../../include/ibdgem_b200.h"
#include "site_math.cuh"

namespace ibdgem {

void set_error(const char *fmt, ...);

#define IBD_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            ::ibdgem::set_error("[::] ERROR in %s (%s:%d): %s", #expr, __FILE__, __LINE__,      \
                                cudaGetErrorString(_e));                                        \
            return 1;                                                                           \
        }                                                                                       \
    } while (0)

// Kernel ids for the per-kernel device timers / launch counters.
enum KernelId {
    K_SITE_TABLE = 0,   // A1 + M3/M4 per-site table
    K_SCAN_COUNT,       // window map: per-block informative-site counts
    K_SCAN_OFFSETS,     // window map: scan of block counts
    K_SCAN_RANK,        // window map: ranks + window first/last sites
    K_WINDOW_NONLD,     // W1/W2 non-LD window log-sums
    K_COUNTERS,         // processed/skipped/final coverage distribution
    K_EXPAND_SITES,     // expanded per-target tab values
    K_LD_GENERAL,       // L1 general CUDA-core --LD window kernel
    K_LD_FINALIZE,      // L2 merge of background-block partial log-sum-exps
    K_LD_COMPACT,       // tensor path: informative sites -> window slots (n, n_ref, l0)
    K_LD_C0,            // tensor path: per-window sum of l0
    K_LD_TRANSPOSE,     // tensor path: site-major bits -> window-padded haplotype-major bits
    K_LD_STAGE,         // tensor path: the call's small tables, read straight from pinned host memory
    K_LD_EXPAND_BG,     // tensor path: background operand (0/1 int8, K-major) + column marginals, keys, Q'
    K_LD_EXPAND_TGT,    // tensor path: target operand (depth-weighted int8, K-major) + row marginals, LIBD2
    K_LD_WINDOWS,       // tensor path: window bookkeeping
    K_LD_IBD0,          // tensor path: LIBD0 log-mean-exp over the background without the target
    K_LD_MMA,           // tensor path: tcgen05 window GEMM + fused log-sum-exp epilogue -> LIBD1
    K_VITERBI,          // H2 hiddengem forward pass (or the whole per-table kernel for small batches)
    K_VITERBI_BACK,     // H3 back-trace + state counts
    K_VITERBI_OUT,      // states back to table-major
    K_FILL,             // NaN fill of device score buffers
    K_V_SLOTS,          // per-target-window tensor path: slots of the K axis (informative kept sites)
    K_V_WMAP,           // -v window map in rank space (one warp per target)
    K_V_TW,             // per (target, window) scalars: C0, R, LIBD2, bookkeeping
    K_V_SORT,           // (target, window) pairs sorted by start, tiles and their K hulls
    K_V_EXPAND_A,       // row operand slabs (n a0, n a1, v nref, v nalt)
    K_V_EXPAND_B,       // column operand slabs (r0, r1, r0 & r1)
    K_LD_VMMA,          // tcgen05 GEMM over per-target windows + fused log-sum-exp -> LIBD0, LIBD1
    K_WINDOW_LINEAR,    // the reference's own running fp64 products per window (ibdgem_scores.w_lik_linear)
    K_POSTERIOR_FWD,    // hiddengem posterior: forward pass, alpha checkpoints per 16-bin chunk
    K_POSTERIOR_BWD,    // hiddengem posterior: backward pass, posteriors + expected occupancy
    K_POSTERIOR_FWD_LOG,  // of the posterior_fwd / _bwd launches, those in natural-log arithmetic (zero or widely
    K_POSTERIOR_BWD_LOG,  // spread penalties); counted only, their time is in posterior_fwd / _bwd
    K_TRACT_COUNT,      // hiddengem tracts: runs of equal state per table, state bytes checked
    K_TRACT_EMIT,       // hiddengem tracts: one 64-byte record per run (likelihood sums, posterior mean / minimum)
    K_POSTERIOR_BWD_MOMENTS,  // hiddengem posterior moments: the backward pass with the covariance recursion (its
                              // forward pass is posterior_fwd; in log arithmetic both are counted under _log too)
    K_POSTERIOR_BWD_TRACTS,   // hiddengem posterior tract counts: the backward pass with the switch sums (and, with the
                              // covariance, its recursion on the solver lane); forward pass and _log counts as above
    K_POSTERIOR_BWD_RUNS,     // hiddengem tract lengths: the backward pass writing per-bin run terms; as above
    K_TRACT_LENGTHS,          // hiddengem tract lengths: windowed run products per start bin and threshold
    K_COUNT
};

extern const char *const *const kKernelNames;  // [K_COUNT], in enum order (engine.cu)

struct LdCache;  // ld_mma.cu
struct VCache;   // ld_vmma.cu

struct PendingTimer {
    int id;
    cudaEvent_t a, b;
};

struct DeviceBuf {
    void *p = nullptr;
    size_t cap = 0;
};

}  // namespace ibdgem

struct ibdgem_engine {
    ibdgem_params prm{};
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    int C = 21;  // max_cov + 1

    // class tables: index = n_ref * C + n_alt
    std::vector<double> h_P;    // [C*C][3]
    std::vector<double> h_lnP;  // [C*C][3]
    double *d_P = nullptr, *d_lnP = nullptr;
    bool depth_linear = false;  // lnP2 - 2 lnP1 + lnP0 == n * kappa for every class
    double kappa = 0, alpha = 0, beta = 0;

    // uploaded inputs
    int64_t S = 0;
    int32_t N = 0;
    int64_t Wh = 0;
    uint64_t *d_pos = nullptr;
    uint8_t *d_nref = nullptr, *d_nalt = nullptr, *d_hostkeep = nullptr;
    double *d_afuser = nullptr;
    uint32_t *d_bits = nullptr;
    bool owns_bits = true;  // false: d_bits is the caller's device buffer (ibdgem_engine_set_panel_device)
    bool have_sites = false, have_panel = false, prepared = false;

    // The panel is copied in site chunks on its own stream; the engine stream waits for a chunk only
    // when a kernel needs its rows, so scoring of the first windows overlaps the rest of the upload.
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_order = nullptr;          // engine stream -> copy stream ordering
    cudaEvent_t ev_book = nullptr;           // window bookkeeping of the current call is final (tensor path)
    // window scores of the tensor path leave for the host range by range while later ranges are still
    // being scored: d2h_stream carries them (copy_stream is busy with the panel chunks)
    cudaStream_t d2h_stream = nullptr;
    std::vector<cudaEvent_t> range_ev;
    std::vector<cudaEvent_t> chunk_ev;       // one per chunk, recorded on copy_stream
    std::vector<int64_t> chunk_end;          // exclusive site end of each chunk
    int chunks_waited = 0;                   // chunks the engine stream already depends on
    int64_t table_from = 0, table_upto = 0;  // site_table has run on [table_from, table_upto)
    // Window shard (multi-GPU, shared windows): this engine scores windows [nW*index/count, nW*(index+1)/count)
    // of every target and touches only the panel rows of those windows (ibdgem_engine_set_window_shard)
    int32_t shard_index = 0, shard_count = 1;
    bool shard_compact = false;              // window shards: the host score table is [T][shard windows][3], not [T][maxW][3]
    bool lazy_table = false;                 // status does not need the panel (no -A, AF range [0, 1])
    std::vector<int64_t> h_wlast;            // host copy of the shared window map (last site per window)

    // prepared, target-independent
    double *d_f = nullptr;
    uint8_t *d_keep = nullptr;    // passes every target-independent filter
    uint8_t *d_status = nullptr;  // shared status (0/1/2)
    double *d_lik7 = nullptr, *d_lnlik7 = nullptr;
    uint32_t *d_rank = nullptr;   // shared exclusive rank of informative sites
    int64_t *d_wfirst = nullptr, *d_wlast = nullptr;  // shared window first/last site
    int32_t *d_nwin_shared = nullptr;  // device copy of nW_shared (window-map view)
    int64_t *d_ktot_shared = nullptr;
    int32_t nW_shared = 0;
    int64_t K_shared = 0;
    // processed / skipped / coverage histogram of a target that -v / -D do not filter ([C + 3], see counters_kernel),
    // accumulated by site_status_kernel in the same pass that decides keep / status (lazy prepare only)
    unsigned long long *d_shared_cnt = nullptr;
    bool shared_cnt_valid = false;

    // tensor path caches (built lazily on first eligible score_ld)
    ibdgem::LdCache *ld = nullptr;
    ibdgem::VCache *vc = nullptr;  // per-target-window tensor path (ld_vmma.cu)

    // scratch
    void *h_pin = nullptr;  // pinned staging for the small per-call host <-> device tables (grow-only)
    size_t h_pin_cap = 0;
    std::vector<ibdgem::DeviceBuf *> scratch;
    int64_t device_bytes = 0;

    // instrumentation
    bool timing = false;
    double k_ms[ibdgem::K_COUNT] = {0};
    int64_t k_launches[ibdgem::K_COUNT] = {0};
    std::vector<ibdgem::PendingTimer> pending;
    std::vector<cudaEvent_t> event_pool;
    // IBDGEM_TIMELINE=<file> (with timing on): every launch, panel chunk and result copy of a step
    // as milliseconds since the step's upload_sites, appended to the file (tools/timeline.py)
    const char *timeline_path = nullptr;
    cudaEvent_t ev_t0 = nullptr, ev_wll = nullptr, ev_bookdone = nullptr;
    bool t0_set = false;

    int64_t hg_flagged = 0;  // tables of the last hiddengem call re-evaluated on the host (near-tie guard)
    int64_t hg_tracts = -1;  // records in SC_HG_TRACTS from the last tract call; -1: none, or that call failed
    int last_ld_path = -1;
    int force_general = 0;
};

namespace ibdgem {

// Timed launch helper: LAUNCH(e, K_ID) { kernel<<<...>>>(...); }
struct LaunchScope {
    ibdgem_engine *e;
    int id;
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s = nullptr;  // the stream the timed work is launched on (default: the engine stream)
    LaunchScope(ibdgem_engine *e_, int id_, cudaStream_t s_ = nullptr);
    ~LaunchScope();
};
int resolve_timers(ibdgem_engine *e);
int settle_timers(ibdgem_engine *e);
// integer value of the environment variable `name` (read by the caller once per process), or dflt when it is unset
inline int env_int(const char *name, int dflt) {
    const char *s = getenv(name);
    return s ? atoi(s) : dflt;
}
// columns of a per-target window map: no target has more windows than S / window_size + 2
inline int map_windows(const ibdgem_engine *e) { return (int)(e->S / e->prm.window_size + 2); }
// Pinned host staging of at least `bytes`.  One buffer: a caller must have synchronised the stream
// that reads or writes it before the next caller asks (every ABI call ends with such a sync).
int pinned_stage(ibdgem_engine *e, size_t bytes, void **out);

// grow-only scratch slots, kept across calls so steady-state scoring does not allocate
enum ScratchSlot {
    SC_TARGETS = 0, SC_BG, SC_TGT_COUNTS, SC_BLOCKCNT, SC_WFIRST, SC_WLAST, SC_NWIN, SC_KTOT, SC_WLL,
    SC_WN, SC_WS, SC_WE, SC_COUNTERS, SC_SITE_STATUS, SC_SITE_LIK, SC_LD_PART, SC_NREFPANEL,
    SC_HG_LIK, SC_HG_OFF, SC_HG_STATE, SC_HG_SCORE, SC_HG_COUNTS, SC_HG_FROMT, SC_HG_LAST,
    SC_MMA_TGT, SC_MMA_BG, SC_MMA_ROWLSE, SC_MMA_BGIDX, SC_MMA_MISC, SC_MMA_UNIT,
    SC_WLIN, SC_WLL_PACK, SC_V_KS, SC_V_KE, SC_V_TWBASE, SC_V_TWI, SC_V_TWD, SC_V_ORDER, SC_V_HIST, SC_V_TILES, SC_V_MISC, SC_HG_CKPT,
    SC_HG_TRACTS,  // the tract records of the last tract call (hiddengem_last_tracts); nothing else writes it
    SC_HG_TOFF, SC_HG_RUNS, SC_HG_RUNSUM, SC_HG_COORD, SC_SLOTS
};
int scratch(ibdgem_engine *e, int slot, size_t bytes, void **out);
// copy_stream with ev_order, and d2h_stream, created on first use (engine.cu)
int side_streams(ibdgem_engine *e);

// hiddengem (hidden.cu): the tables of one call.  Table t holds len(t) bins from bin start(t) of every per-bin array:
// start(t) = bin_offsets[t] (packed, table_stride = 0) or t * table_stride.
struct HgCall {
    int n = 0;
    std::vector<int64_t> sl;  // [n] starts, then [n] lengths
    int64_t maxbins = 0, total = 0;
    int64_t *d_start = nullptr, *d_len = nullptr;  // the same in device memory (SC_HG_OFF)
    int64_t start(int t) const { return sl[(size_t)t]; }
    int64_t len(int t) const { return sl[(size_t)n + t]; }
};
// The prologue of every hiddengem entry: the layout (1 and the error set on a negative length or one past the
// stride; with need_bins, also when the call has no bins), the engine's device, and start / length uploaded on the
// engine stream.
int hg_begin(ibdgem_engine *e, const char *fn, int n_tables, const int64_t *bin_offsets, int64_t table_stride, bool need_bins,
             HgCall *c);
// Scratch of a Viterbi pass over nb host bins: likelihoods, scores (nb x 24 B), states and, behind them, the per-table
// near-tie flags (d_flag = d_state + nb), and counts.  The posterior pass may reuse SC_HG_SCORE and SC_HG_COUNTS (the
// tract entry runs it after the Viterbi pass); nothing but the Viterbi pass writes SC_HG_STATE.
struct HgViterbiScratch {
    double *lik, *score;
    uint8_t *state, *flag;
    long long *counts;
};
int viterbi_scratch(ibdgem_engine *e, int n_tables, int64_t nb, HgViterbiScratch *s);
// Viterbi kernels for one batch of tables in device memory; no host synchronisation.  d_flag[t] = 1 marks a table the
// near-tie guard hands to the host.
int viterbi_on_device(ibdgem_engine *e, int n_tables, int64_t maxbins, int64_t total_bins, const int64_t *d_start, const int64_t *d_len,
                      const double *d_lik, int is_log, double p01, double p02, double p12, uint8_t *d_state, double *d_score,
                      long long *d_counts, uint8_t *d_flag);
// The near-tie guard's verdict: the tables with h_flag[t] != 0 re-evaluated in long double on a few host threads, and
// e->hg_flagged set to their number.  Table t is read at bin c.start(t) of lik (device memory when lik_on_device) and
// its states, scores and counts are written to the same places of state, score and counts (each may be null; device
// memory when out_on_device, written on the engine stream, which is then synchronised).
int viterbi_resolve(ibdgem_engine *e, const HgCall &c, const std::vector<uint8_t> &h_flag, const double *lik, bool lik_on_device,
                    int is_log, double p01, double p02, double p12, uint8_t *state, double *score, int64_t *counts, bool out_on_device);
// posterior.cu: penalty check of the posterior entries (1 and the error set when rejected), and its kernels for one
// batch of tables in device memory (no host synchronisation).  d_cov != null runs the moment variant of the backward
// pass: covariances into d_cov [n_tables][3][3], and d_post may then be null.  d_sw != null runs the tract-count
// variant instead: switches into d_sw [n_tables][3][3], tract counts into d_tr [n_tables][3], their covariance into
// d_cov when that is not null; d_post is then not written.  d_runs != null runs the run-term variant instead: gamma,
// d and ln c of every bin into d_runs [bin][9] in the layout of d_lik; d_post is then not written.
bool bad_penalties(const char *fn, double p01, double p02, double p12);
int posterior_on_device(ibdgem_engine *e, int n_tables, int64_t maxbins, const int64_t *d_start, const int64_t *d_len, const double *d_lik,
                        int is_log, double p01, double p02, double p12, double *d_post, double *d_expected, double *d_cov = nullptr,
                        double *d_sw = nullptr, double *d_tr = nullptr, double *d_runs = nullptr);

// Makes the engine stream wait for the panel chunks that cover sites [0, s_end); ensure_table also
// runs site_table on the part of [0, s_end) it has not covered yet.
int wait_panel_upto(ibdgem_engine *e, int64_t s_end);
int ensure_table(ibdgem_engine *e, int64_t s_end);

int dev_alloc(ibdgem_engine *e, void **p, size_t bytes);
void dev_free(ibdgem_engine *e, void *p, size_t bytes);

// The call's background as both tensor paths see it (ld_mma.cu): the unique individuals in ascending order with
// ln(multiplicity) — the pileup's own individual never contributes (src/ibdgem.c:714) — and per target its own index in
// that list (-1: none) and nb, the background size without it, with ln nb (NaN when nb = 0: 0/0 in the reference).
struct LdBackground {
    std::vector<int32_t> bgU;
    std::vector<double> lnc;
    std::vector<int32_t> own;
    std::vector<int32_t> nb;
    std::vector<double> lognb;
};
void ld_background(int32_t N, int32_t T, const int32_t *h_targets, int32_t n_bg, const int32_t *h_bg, int32_t pu_idx, LdBackground *out);

// The scoring paths of score_ld / score_nonld; ibdgem_engine_last_ld_path reports the --LD one that ran.
enum ScorePath { NONLD = -1, LD_GENERAL = 0, LD_TENSOR = 1, LD_VTENSOR = 2 };

// One scoring call: its inputs, the window outputs in device memory, the caller's destinations of the window scores,
// and the copies into them that a tensor path has already issued (the call's end waits for exactly those streams).
struct ScoreCall {
    int32_t T = 0;
    const int32_t *d_targets = nullptr;  // [T]
    SiteView v{};                        // v.tgt_counts: the call's -D counts in device memory, [T][S][2], or nullptr
    LdBackground bg;                     // --LD
    int32_t outW = 0;                    // columns of the window outputs
    double *d_wll = nullptr;             // [T][outW][3]
    int32_t *d_wn = nullptr;             // [T][outW]
    uint64_t *d_ws = nullptr, *d_we = nullptr;  // [T][outW]
    int32_t *d_nwout = nullptr;          // [T]
    double *w_loglik = nullptr;          // the caller's host table [T][outW][3], or nullptr
    double *w_loglik_device = nullptr;   // the caller's device table (may be peer memory), or nullptr
    bool streamed = false;               // the copies of d_wll to w_loglik are issued on d2h_stream
    bool dev_streamed = false;           // the copies of d_wll to w_loglik_device are issued on d2h_stream
    bool bookkeeping_ready = false;      // ev_book is recorded: the bookkeeping copies may go on copy_stream
};

// tensor-path entry points (ld_mma.cu)
bool ld_tensor_eligible(ibdgem_engine *e, int32_t n_targets, int32_t n_bg, const uint8_t *tgt_counts);
int ld_tensor_prepare(ibdgem_engine *e);
int ld_tensor_score(ibdgem_engine *e, ScoreCall &c);
void ld_tensor_release(ibdgem_engine *e);
constexpr int PANEL_CHUNKS = 16;         // upload / scoring pipeline depth
constexpr size_t PANEL_CHUNK_MIN_BYTES = (size_t)16 << 20;  // ~0.3 ms of PCIe; smaller panels use fewer chunks
void ld_tensor_invalidate(ibdgem_engine *e);
// site-major bits -> [block][haplotype][WP32 words] for `nwin` blocks of Wpad slots listed in `infsite` (ld_mma.cu)
int ld_transpose_launch(ibdgem_engine *e, int w_begin, int w_end, const int32_t *infsite, int Wpad, int WP32, int H, uint32_t *tbits);
// device alias of the caller's host table c.w_loglik when it is page-locked and mapped, else nullptr (ld_mma.cu)
double *host_table_alias(const ScoreCall &c);
// *ev = e->range_ev[k], creating the events up to k as needed (ld_mma.cu)
int range_event(ibdgem_engine *e, size_t k, cudaEvent_t *ev);
// per-target-window tensor path (ld_vmma.cu): -v / -D; nU is the size of the call's unique background
bool ld_vtensor_eligible(ibdgem_engine *e, int32_t n_targets, int32_t nU);
int ld_vtensor_score(ibdgem_engine *e, ScoreCall &c);
void ld_vtensor_release(ibdgem_engine *e);
void ld_vtensor_invalidate(ibdgem_engine *e);
// window map for `rows` rows (targets == nullptr: one shared row), engine.cu
int build_window_map(ibdgem_engine *e, const SiteView &v, const int32_t *d_targets, int rows, int maxW, int64_t *d_wfirst,
                     int64_t *d_wlast, int32_t *d_nwin, int64_t *d_ktot, uint32_t *d_rank);
// windows [w_begin, w_end) and panel rows [s_begin, s_end) of this engine's shard (everything when unsharded)
void window_shard_bounds(const ibdgem_engine *e, int32_t *w_begin, int32_t *w_end, int64_t *s_begin, int64_t *s_end);

}  // namespace ibdgem
