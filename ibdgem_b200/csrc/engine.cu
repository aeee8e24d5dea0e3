// engine.cu — C ABI of libibdgem_b200.so, host orchestration, and the general CUDA-core kernels:
// per-site table (A1, M3-M5), window map (W2), non-LD window log-sums (W1), counters (F1),
// expanded tab values, and the general --LD window kernel (L1, L2) that handles every mode
// (-v, -D, arbitrary class tables).  The tensor-core --LD path lives in ld_mma.cu, the batched
// hiddengem Viterbi in hidden.cu.  Reference citations are relative to /root/reference.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "engine.h"
#include "site_math.cuh"

namespace ibdgem {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

static const char *const kKernelNameList[] = {
    "site_table",     "scan_count",    "scan_offsets",  "scan_rank",    "window_nonld", "counters",
    "expand_sites",   "ld_general",    "ld_finalize",   "ld_compact",   "ld_c0",        "ld_transpose",
    "ld_stage",       "ld_expand_bg",  "ld_expand_tgt", "ld_windows",   "ld_ibd0",
    "ld_mma",         "viterbi",       "viterbi_back",  "viterbi_out",  "fill",
    "v_slots",        "v_wmap",        "v_tw",          "v_sort",       "v_expand_a",  "v_expand_b",   "ld_vmma",
    "window_linear",  "posterior_fwd", "posterior_bwd", "posterior_fwd_log", "posterior_bwd_log",
    "tract_count",    "tract_emit",    "posterior_bwd_moments",
};
static_assert(sizeof(kKernelNameList) / sizeof(kKernelNameList[0]) == K_COUNT, "one name per KernelId, in enum order");
const char *const *const kKernelNames = kKernelNameList;

// ---------------------------------------------------------------------------------------------
// instrumentation
LaunchScope::LaunchScope(ibdgem_engine *e_, int id_, cudaStream_t s_) : e(e_), id(id_), s(s_ ? s_ : e_->stream) {
    e->k_launches[id]++;
    if (!e->timing) return;
    auto get = [&]() {
        cudaEvent_t ev;
        if (!e->event_pool.empty()) {
            ev = e->event_pool.back();
            e->event_pool.pop_back();
        } else {
            cudaEventCreate(&ev);
        }
        return ev;
    };
    a = get();
    b = get();
    cudaEventRecord(a, s);
}
LaunchScope::~LaunchScope() {
    if (!a) return;
    cudaEventRecord(b, s);
    e->pending.push_back({id, a, b});
}
// End of an ABI call: the event pairs of its launches stay pending — they are read when somebody asks for the statistics
// (kernel_stats / reset_stats), when a timeline is being written, or when many have piled up.  Reading them at the end of
// every call cost ~0.3 ms of host time per call (two driver calls per launch), which the next call then started late by.
int settle_timers(ibdgem_engine *e) {
    if (e->t0_set || e->pending.size() > 4096) return resolve_timers(e);
    return 0;
}
int resolve_timers(ibdgem_engine *e) {
    FILE *tl = e->timeline_path && e->t0_set && !e->pending.empty() ? fopen(e->timeline_path, "a") : nullptr;
    for (auto &p : e->pending) {
        float ms = 0;
        cudaEventSynchronize(p.b);
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) e->k_ms[p.id] += ms;
        if (tl) {
            float t_a = 0, t_b = 0;
            cudaEventElapsedTime(&t_a, e->ev_t0, p.a);
            cudaEventElapsedTime(&t_b, e->ev_t0, p.b);
            fprintf(tl, "%s %.4f %.4f\n", kKernelNames[p.id], t_a, t_b);
        }
        e->event_pool.push_back(p.a);
        e->event_pool.push_back(p.b);
    }
    e->pending.clear();
    if (tl) fclose(tl);
    return 0;
}

int dev_alloc(ibdgem_engine *e, void **p, size_t bytes) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    IBD_CUDA(cudaMalloc(p, bytes));
    e->device_bytes += (int64_t)bytes;
    return 0;
}
void dev_free(ibdgem_engine *e, void *p, size_t bytes) {
    if (!p) return;
    cudaFree(p);
    e->device_bytes -= (int64_t)(bytes ? bytes : 16);
}

int pinned_stage(ibdgem_engine *e, size_t bytes, void **out) {
    if (e->h_pin_cap < bytes) {
        if (e->h_pin) cudaFreeHost(e->h_pin);
        e->h_pin = nullptr;
        e->h_pin_cap = 0;
        const size_t want = bytes + bytes / 4 + 4096;
        IBD_CUDA(cudaMallocHost(&e->h_pin, want));
        e->h_pin_cap = want;
    }
    *out = e->h_pin;
    return 0;
}

int scratch(ibdgem_engine *e, int slot, size_t bytes, void **out) {
    if (e->scratch.empty()) e->scratch.assign(SC_SLOTS, nullptr);
    DeviceBuf *&b = e->scratch[slot];
    if (!b) b = new DeviceBuf();
    if (b->cap < bytes) {
        if (b->p) dev_free(e, b->p, b->cap);
        b->p = nullptr;
        b->cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        if (dev_alloc(e, &b->p, want)) return 1;
        b->cap = want;
    }
    *out = b->p;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// device helpers
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void fill_nan_kernel(double *p, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = nan;
}

// ---------------------------------------------------------------------------------------------
// K_SITE_TABLE: a warp takes 32 consecutive panel lines.  Phase 1 streams the packed rows with
// 128-bit loads (four lanes per row) and popcounts them for the allele frequency (find_f_impute,
// src/ibd-parse.c:91-99); lane r ends up with row r's count.  Phase 2 is lane-parallel, one site per
// lane: the AF-range and max-cov filters (src/ibdgem.c:616-626), IBD0, IBD1|g, IBD2|g
// (src/ibd-math.c:84-142, src/ibdgem.c:632-651) and their logs.
__global__ void __launch_bounds__(256)
site_table_kernel(int64_t s_begin, int64_t S, int32_t N, int64_t Wh, const uint32_t *__restrict__ bits,
                  const uint8_t *__restrict__ hostkeep, const uint8_t *__restrict__ nref,
                  const uint8_t *__restrict__ nalt, const double *__restrict__ afuser,
                  const double *__restrict__ Ptab, int C, double min_af, double max_af, int max_cov,
                  double *__restrict__ f_out, uint8_t *__restrict__ keep, uint8_t *__restrict__ status,
                  double *__restrict__ lik7, double *__restrict__ lnlik7, const double *__restrict__ lnPtab) {
    __shared__ double stage7[8][32 * 7];
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int H = 2 * N;
    const int nfull = H >> 5, rem = H & 31;
    const bool vec4 = ((Wh & 3) == 0);
    const int n4 = vec4 ? (nfull >> 2) : 0;
    for (int64_t s0 = s_begin + warp0 * 32; s0 < S; s0 += nwarps * 32) {  // S = exclusive end of the range
        const int rows = (int)min((int64_t)32, S - s0);
        // four lanes share a row (eight rows per pass): ten independent 16-byte loads per lane, two
        // shuffles to join the quarters, one to hand row r's count to lane r
        int mycnt = 0;
        const int j = lane >> 2, q = lane & 3;
#pragma unroll
        for (int it = 0; it < 4; it++) {
            const int r = it * 8 + j;
            int cnt = 0;
            if (r < rows) {
                const uint32_t *row = bits + (s0 + r) * Wh;
                const uint4 *row4 = reinterpret_cast<const uint4 *>(row);
                for (int w = q; w < n4; w += 4) {
                    const uint4 x = __ldg(row4 + w);
                    cnt += __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
                }
                for (int w = (n4 << 2) + q; w < nfull; w += 4) cnt += __popc(__ldg(row + w));
                if (q == 0 && rem) cnt += __popc(__ldg(row + nfull) & ((1u << rem) - 1u));
            }
            cnt += __shfl_xor_sync(0xffffffffu, cnt, 1);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, 2);
            const int got = __shfl_sync(0xffffffffu, cnt, 4 * (lane & 7));
            if ((lane >> 3) == it) mycnt = got;
        }
        const int64_t s = s0 + lane;
        double v[7], lv[7];
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
        for (int i = 0; i < 7; i++) v[i] = lv[i] = nan;
        if (lane < rows) {
            double f = __ddiv_rn((double)mycnt, (double)H);
            if (afuser) {
                const double u = afuser[s];
                if (u == u) f = u;  // src/ibdgem.c:609-614
            }
            const int r = nref[s], a = nalt[s];
            const bool k = hostkeep[s] && !(f > max_af || f < min_af) && (r + a <= max_cov);
            if (k) {
                const double *P = Ptab + (size_t)(r * C + a) * 3;
                const double P0 = P[0], P1 = P[1], P2 = P[2];
                v[0] = lik_ibd0(f, P0, P1, P2);
                v[1] = lik_ibd1(0, f, P0, P1, P2);
                v[2] = lik_ibd1(1, f, P0, P1, P2);
                v[3] = lik_ibd1(2, f, P0, P1, P2);
                v[4] = P0; v[5] = P1; v[6] = P2;
            }
            // ln P(D | g) comes from the engine's table (the long double logarithms every other path uses): three of the
            // seven fp64 logarithms of a site
            const double *lP = lnPtab + (k ? (size_t)(r * C + a) * 3 : 0);
#pragma unroll
            for (int i = 0; i < 7; i++) lv[i] = k ? (i >= 4 ? lP[i - 4] : log(v[i])) : v[i];
            f_out[s] = f;
            keep[s] = k ? 1 : 0;
            status[s] = k ? ((r + a >= 1) ? 1 : 2) : 0;
        }
        // the warp's 32 x 7 values of each table are contiguous in memory: they pass through shared memory so that every
        // store instruction writes 256 contiguous bytes (a lane storing its own seven doubles touched 14 lines per
        // instruction — ncu: the table half of this kernel was bound by those stores)
        double *stw = stage7[threadIdx.x >> 5];
#pragma unroll
        for (int pass = 0; pass < 2; pass++) {
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 7; i++) stw[lane * 7 + i] = pass ? lv[i] : v[i];
            __syncwarp();
            double *dst = (pass ? lnlik7 : lik7) + s0 * 7;
            for (int i = lane; i < rows * 7; i += 32) dst[i] = stw[i];
        }
    }
}

// Site status without the panel: when no -A table is given and the AF range is the default [0, 1]
// the AF filter of src/ibdgem.c:616 cannot fire (f = count / 2N), so keep / status follow from the
// site arrays alone and the window map can be built before the panel has arrived.
// The same pass accumulates the counters of a target that -v / -D do not filter (processed, skipped, total
// final coverage, coverage histogram: src/ibdgem.c:585-630, 761-768) — one read of the site arrays instead of two.
__global__ void __launch_bounds__(256)
site_status_kernel(int64_t S, const uint8_t *__restrict__ hostkeep, const uint8_t *__restrict__ nref,
                   const uint8_t *__restrict__ nalt, int max_cov, uint8_t *__restrict__ keep, uint8_t *__restrict__ status,
                   int C, unsigned long long *__restrict__ cnt /*[C+3], pre-zeroed*/) {
    extern __shared__ unsigned int shist[];  // [C + 3]: a block sees at most 2^32 - 1 sites
    for (int i = threadIdx.x; i < C + 3; i += blockDim.x) shist[i] = 0;
    __syncthreads();
    unsigned proc = 0, skip = 0, cov = 0;
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < S; s += (int64_t)gridDim.x * blockDim.x) {
        const int r = nref[s], a = nalt[s];
        const bool k = hostkeep[s] && (r + a <= max_cov);
        keep[s] = k ? 1 : 0;
        status[s] = k ? ((r + a >= 1) ? 1 : 2) : 0;
        if (k) {
            proc++;
            cov += (unsigned)(r + a);
            atomicAdd(&shist[3 + min(r + a, C - 1)], 1u);
        } else {
            skip++;
        }
    }
    proc = (unsigned)warp_sum_i((int)proc);
    skip = (unsigned)warp_sum_i((int)skip);
    cov = (unsigned)warp_sum_i((int)cov);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&shist[0], proc);
        atomicAdd(&shist[1], skip);
        atomicAdd(&shist[2], cov);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C + 3; i += blockDim.x)
        if (shist[i]) atomicAdd(&cnt[i], (unsigned long long)shist[i]);
}

// ---------------------------------------------------------------------------------------------
// Window map (W2, src/ibdgem.c:559-578, 723-730): windows are runs of `window` informative kept
// sites in file order.  Three small kernels: per-block counts, scan of block counts, and a
// ranked pass that records the first and last site of every window.  Rows = 1 (shared map) or
// one per target (-v / -D make the kept set target-dependent).
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITERS = 8;
constexpr int SCAN_CHUNK = SCAN_THREADS * SCAN_ITERS;
constexpr int ROW_SLICE = 32768;  // target rows per launch where they ride on gridDim.y

__global__ void __launch_bounds__(SCAN_THREADS)
scan_count_kernel(SiteView v, const int32_t *__restrict__ targets, uint32_t *__restrict__ blockcnt,
                  int nb) {
    const int t = blockIdx.y;
    const int indiv = targets ? targets[t] : 0;
    const int64_t base = (int64_t)blockIdx.x * SCAN_CHUNK;
    int c = 0;
    for (int it = 0; it < SCAN_ITERS; it++) {
        const int64_t s = base + it * SCAN_THREADS + threadIdx.x;
        int r, a, g;
        if (s < v.S && site_eval(v, t, indiv, s, r, a, g) == 1) c++;
    }
    c = warp_sum_i(c);
    __shared__ int ws[SCAN_THREADS / 32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int i = 0; i < SCAN_THREADS / 32; i++) tot += ws[i];
        blockcnt[(int64_t)t * nb + blockIdx.x] = tot;
    }
}

// one block per row: exclusive scan of that row's block counts (in place), total -> ktot, nwin
__global__ void __launch_bounds__(256)
scan_offsets_kernel(uint32_t *__restrict__ blockcnt, int nb, int window, int64_t *__restrict__ ktot,
                    int32_t *__restrict__ nwin) {
    const int t = blockIdx.x;
    uint32_t *row = blockcnt + (int64_t)t * nb;
    __shared__ uint32_t carry;
    __shared__ uint32_t ws[8];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nb; b0 += 256) {
        const int i = b0 + threadIdx.x;
        const uint32_t v = (i < nb) ? row[i] : 0;
        uint32_t x = v;  // inclusive warp scan
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31) >= o) x += y;
        }
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
        __syncthreads();
        uint32_t woff = 0;
        for (int w = 0; w < (int)(threadIdx.x >> 5); w++) woff += ws[w];
        const uint32_t excl = carry + woff + x - v;
        if (i < nb) row[i] = excl;
        __syncthreads();
        if (threadIdx.x == 255) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        ktot[t] = carry;
        nwin[t] = (int32_t)((carry + (uint32_t)window - 1) / (uint32_t)window);
    }
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_rank_kernel(SiteView v, const int32_t *__restrict__ targets, const uint32_t *__restrict__ blockoff,
                 int nb, int window, const int64_t *__restrict__ ktot, int64_t *__restrict__ wfirst,
                 int64_t *__restrict__ wlast, int maxW, uint32_t *__restrict__ rank_out) {
    const int t = blockIdx.y;
    const int indiv = targets ? targets[t] : 0;
    const int64_t base = (int64_t)blockIdx.x * SCAN_CHUNK;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __shared__ int ws[SCAN_THREADS / 32];
    uint32_t running = blockoff[(int64_t)t * nb + blockIdx.x];
    const int64_t K = ktot[t];
    for (int it = 0; it < SCAN_ITERS; it++) {
        const int64_t s = base + it * SCAN_THREADS + threadIdx.x;
        int r, a, g;
        const bool inf = (s < v.S) && site_eval(v, t, indiv, s, r, a, g) == 1;
        const uint32_t bal = __ballot_sync(0xffffffffu, inf);
        if (lane == 0) ws[wid] = __popc(bal);
        __syncthreads();
        uint32_t off = running;
        int tot = 0;
        for (int w = 0; w < SCAN_THREADS / 32; w++) {
            if (w < wid) off += ws[w];
            tot += ws[w];
        }
        const uint32_t rk = off + __popc(bal & ((1u << lane) - 1u));
        if (rank_out && s < v.S) rank_out[s] = rk;
        if (inf) {
            const uint32_t w = rk / (uint32_t)window, k = rk % (uint32_t)window;
            if ((int)w < maxW) {
                if (k == 0) wfirst[(int64_t)t * maxW + w] = s;
                if (k == (uint32_t)window - 1 || (int64_t)rk == K - 1) wlast[(int64_t)t * maxW + w] = s;
            }
        }
        running += tot;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// K_WINDOW_NONLD: one warp per (target, window).  Sums ln IBD0, ln IBD1, ln IBD2 over the
// informative sites of the window (the products of src/ibdgem.c:665-667 in log space) and emits
// the window bookkeeping (src/ibdgem.c:723-730, 736, 751-756).
struct WindowMapView {
    const int64_t *wfirst, *wlast;
    const int32_t *nwin;
    int rows;  // 1 = shared
    int maxW;
};

__global__ void __launch_bounds__(256)
window_nonld_kernel(SiteView v, WindowMapView m, const int32_t *__restrict__ targets, int T,
                    const uint64_t *__restrict__ pos, const double *__restrict__ f,
                    const double *__restrict__ lnlik7, const double *__restrict__ Ptab, int C,
                    int outW, double *__restrict__ wll, int32_t *__restrict__ wn,
                    uint64_t *__restrict__ ws, uint64_t *__restrict__ we, int32_t *__restrict__ nwin_out) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t total = (int64_t)T * outW;
    if (gw >= total) return;
    const int t = (int)(gw / outW), w = (int)(gw % outW);
    const int row = (m.rows == 1) ? 0 : t;
    const int nw = m.nwin[row];
    if (w == 0 && lane == 0) nwin_out[t] = nw;
    if (w >= nw || w >= m.maxW) return;
    const int indiv = targets[t];
    const int64_t s0 = m.wfirst[(int64_t)row * m.maxW + w], s1 = m.wlast[(int64_t)row * m.maxW + w];
    double a0 = 0, a1 = 0, a2 = 0;
    int n = 0;
    for (int64_t s = s0 + lane; s <= s1; s += 32) {
        int r, a, g;
        if (site_eval(v, t, indiv, s, r, a, g) != 1) continue;
        n++;
        if (v.tgt_counts) {  // -D: per-target counts, evaluate the closed forms here
            const double *P = Ptab + (size_t)(r * C + a) * 3;
            const double P0 = P[0], P1 = P[1], P2 = P[2], ff = f[s];
            a0 += log(lik_ibd0(ff, P0, P1, P2));
            a1 += log(lik_ibd1(g, ff, P0, P1, P2));
            a2 += log(P[g]);
        } else {
            const double *L = lnlik7 + s * 7;
            a0 += L[0];
            a1 += L[1 + g];
            a2 += L[4 + g];
        }
    }
    a0 = warp_sum_d(a0);
    a1 = warp_sum_d(a1);
    a2 = warp_sum_d(a2);
    n = warp_sum_i(n);
    if (lane == 0) {
        const int64_t o = (int64_t)t * outW + w;
        wll[o * 3 + 0] = a0;
        wll[o * 3 + 1] = a1;
        wll[o * 3 + 2] = a2;
        wn[o] = n;
        ws[o] = pos[s0];
        we[o] = pos[s1];
    }
}

// K_WINDOW_NONLD, shared window map (no -v, no -D): one CTA per window, one thread per target.
// The window's rows of the per-site log table (56 bytes per site, target-independent) are staged
// in shared memory once per CTA; every thread then walks the sites with its target's genotype
// bits, so the table is read from HBM once per window instead of once per target.  The kernel is
// issue-bound (ncu: 68 % issue slots, 19 % L2), so the walk is kept short: the row offset of every
// staged site is precomputed, ln IBD1 | g and ln IBD2 | g of a site sit side by side (one 16-byte
// shared load per site and target), and LIBD0 — the same for every target — is summed once per CTA
// from the values the threads stage.
constexpr int NONLD_TILE = 256;  // sites staged per pass
template <int NONLD_BATCH>  // genotype loads in flight per thread
__global__ void __launch_bounds__(128)
window_nonld_shared_kernel(SiteView v, WindowMapView m, const int32_t *__restrict__ targets, int T,
                           const uint64_t *__restrict__ pos, const uint8_t *__restrict__ status,
                           const double *__restrict__ lnlik7, int outW, double *__restrict__ wll,
                           int32_t *__restrict__ wn, uint64_t *__restrict__ ws, uint64_t *__restrict__ we,
                           int32_t *__restrict__ nwin_out) {
    __shared__ double2 sl12[NONLD_TILE][3];  // [site][g] = (ln IBD1 | g, ln IBD2 | g)
    __shared__ int64_t srow[NONLD_TILE];     // word offset of the site's panel line
    __shared__ int32_t soff[NONLD_TILE];     // the site, relative to the window's first
    __shared__ int segcnt[NONLD_TILE / 32];
    __shared__ double sa0[4];
    constexpr int PASSES = NONLD_TILE / 128;
    const int w = blockIdx.x;
    const int nw = m.nwin[0];
    const int t = blockIdx.y * blockDim.x + threadIdx.x;
    if (w == 0 && t < T) nwin_out[t] = nw;
    if (w >= nw || w >= m.maxW) return;
    const int64_t s0 = m.wfirst[w], s1 = m.wlast[w];
    const int indiv = t < T ? targets[t] : 0;
    const uint32_t *tcol = v.bits + (indiv >> 4);
    const int tsh = (indiv & 15) * 2;
    const int lane = threadIdx.x & 31;
    double a0p = 0, a1 = 0, a2 = 0;  // a0p: this thread's share of the window's LIBD0 terms
    int n = 0;
    for (int64_t sb = s0; sb <= s1; sb += NONLD_TILE) {
        __syncthreads();
        // compact the informative sites of this pass into shared memory, in site order
        unsigned bal[PASSES];
#pragma unroll
        for (int q = 0; q < PASSES; q++) {
            const int64_t s = sb + q * 128 + threadIdx.x;
            bal[q] = __ballot_sync(0xffffffffu, s <= s1 && status[s] == 1);
            if (lane == 0) segcnt[(q * 128 + threadIdx.x) >> 5] = __popc(bal[q]);
        }
        __syncthreads();
        int cnt = 0;
#pragma unroll
        for (int q = 0; q < PASSES; q++) {
            const int seg = (q * 128 + (int)threadIdx.x) >> 5;
            int base = 0;
            for (int k = 0; k < seg; k++) base += segcnt[k];
            if ((bal[q] >> lane) & 1u) {
                const int slot = base + __popc(bal[q] & ((1u << lane) - 1u));
                const int64_t site = sb + q * 128 + threadIdx.x;
                srow[slot] = site * v.Wh;
                soff[slot] = (int32_t)(site - s0);
            }
        }
        for (int k = 0; k < NONLD_TILE / 32; k++) cnt += segcnt[k];
        __syncthreads();
        for (int i = threadIdx.x; i < cnt * 7; i += blockDim.x) {
            const int j = i / 7, c = i - j * 7;
            const double x = lnlik7[(s0 + soff[j]) * 7 + c];
            double *dst = reinterpret_cast<double *>(&sl12[j][0]);
            if (c == 0)
                a0p += x;
            else if (c <= 3)
                dst[(c - 1) * 2] = x;
            else
                dst[(c - 4) * 2 + 1] = x;
        }
        __syncthreads();
        if (t < T) {
            // genotype loads are issued NONLD_BATCH at a time: one dependent global load per site made this loop a
            // chain of L2 round trips
            for (int j0 = 0; j0 < cnt; j0 += NONLD_BATCH) {
                uint32_t pr[NONLD_BATCH];
#pragma unroll
                for (int q = 0; q < NONLD_BATCH; q++) pr[q] = (j0 + q < cnt) ? __ldg(tcol + srow[j0 + q]) : 0u;
#pragma unroll
                for (int q = 0; q < NONLD_BATCH; q++) {
                    if (j0 + q < cnt) {
                        const int g = __popc((pr[q] >> tsh) & 3u);
                        const double2 l = sl12[j0 + q][g];
                        a1 += l.x;
                        a2 += l.y;
                    }
                }
            }
            n += cnt;
        }
    }
    // LIBD0 of the window: the threads' shares, joined once
    a0p = warp_sum_d(a0p);
    if (lane == 0) sa0[threadIdx.x >> 5] = a0p;
    __syncthreads();
    if (t < T) {
        const double a0 = (sa0[0] + sa0[1]) + (sa0[2] + sa0[3]);
        const int64_t o = (int64_t)t * outW + w;
        wll[o * 3 + 0] = a0;
        wll[o * 3 + 1] = a1;
        wll[o * 3 + 2] = a2;
        wn[o] = n;
        ws[o] = pos[s0];
        we[o] = pos[s1];
    }
}

// K_WINDOW_LINEAR: the reference's own window aggregates, bit for bit — one thread per (target, window) multiplies
// the per-site likelihoods in file order with round-to-nearest fp64 products starting from 1.0, exactly the sequence
// of src/ibdgem.c:562, 665-667 (no fused operations, no reassociation), so denormals and the underflow to 0 come out
// as they do there.  The per-site values themselves are the reference's doubles (tab.txt columns, tested).
__global__ void __launch_bounds__(128)
window_linear_kernel(SiteView v, WindowMapView m, const int32_t *__restrict__ targets, int T, const double *__restrict__ f,
                     const double *__restrict__ lik7, const double *__restrict__ Ptab, int C, int outW, double *__restrict__ wlin) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * outW) return;
    const int t = (int)(i / outW), w = (int)(i % outW);
    const int row = (m.rows == 1) ? 0 : t;
    if (w >= m.nwin[row] || w >= m.maxW) return;
    const int indiv = targets[t];
    const int64_t s0 = m.wfirst[(int64_t)row * m.maxW + w], s1 = m.wlast[(int64_t)row * m.maxW + w];
    double p0 = 1.0, p1 = 1.0, p2 = 1.0;
    for (int64_t s = s0; s <= s1; s++) {
        int r, a, g;
        if (site_eval(v, t, indiv, s, r, a, g) != 1) continue;
        double l0, l1, l2;
        if (v.tgt_counts) {
            const double *P = Ptab + (size_t)(r * C + a) * 3;
            l0 = lik_ibd0(f[s], P[0], P[1], P[2]);
            l1 = lik_ibd1(g, f[s], P[0], P[1], P[2]);
            l2 = P[g];
        } else {
            const double *L = lik7 + s * 7;
            l0 = L[0];
            l1 = L[1 + g];
            l2 = L[4 + g];
        }
        p0 = __dmul_rn(p0, l0);
        p1 = __dmul_rn(p1, l1);
        p2 = __dmul_rn(p2, l2);
    }
    wlin[i * 3 + 0] = p0;
    wlin[i * 3 + 1] = p1;
    wlin[i * 3 + 2] = p2;
}

// ---------------------------------------------------------------------------------------------
// K_COUNTERS: processed / skipped / final coverage histogram per target (src/ibdgem.c:537-545,
// 585-630, 734, 761-768).  grid = (site chunks, rows); shared-memory histogram per block, then
// 64-bit integer atomics into the row's (pre-zeroed) counters, so the result is exact.
constexpr int COUNTERS_CHUNK = 8192;
__global__ void __launch_bounds__(256)
counters_kernel(SiteView v, const int32_t *__restrict__ targets, int C,
                unsigned long long *__restrict__ out /*[rows][C+3]*/) {
    const int t = blockIdx.y;
    const int indiv = targets ? targets[t] : 0;
    extern __shared__ unsigned long long sh[];  // [C+3]
    for (int i = threadIdx.x; i < C + 3; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    unsigned long long proc = 0, skip = 0, cov = 0;
    const int64_t s_begin = (int64_t)blockIdx.x * COUNTERS_CHUNK;
    const int64_t s_end = min(v.S, s_begin + COUNTERS_CHUNK);
    for (int64_t s = s_begin + threadIdx.x; s < s_end; s += blockDim.x) {
        int r = 0, a = 0, g = 0;
        const int st = site_eval(v, t, indiv, s, r, a, g);
        if (st == 0) {
            skip++;
        } else {
            proc++;
            cov += (unsigned)(r + a);
            atomicAdd(&sh[3 + min(r + a, C - 1)], 1ULL);
        }
    }
    atomicAdd(&sh[0], proc);
    atomicAdd(&sh[1], skip);
    atomicAdd(&sh[2], cov);
    __syncthreads();
    for (int i = threadIdx.x; i < C + 3; i += blockDim.x)
        if (sh[i]) atomicAdd(&out[(int64_t)t * (C + 3) + i], sh[i]);
}

// K_EXPAND_SITES: the LIBD0/LIBD1/LIBD2 columns of every tab.txt row (src/ibdgem.c:641-663,
// 731-733), one thread per (target, site), coalesced stores.
__global__ void __launch_bounds__(256)
expand_sites_kernel(SiteView v, const int32_t *__restrict__ targets, int T,
                    const double *__restrict__ f, const double *__restrict__ lik7,
                    const double *__restrict__ Ptab, int C, uint8_t *__restrict__ st_out,
                    double *__restrict__ lik_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * v.S) return;
    const int t = (int)(i / v.S);
    const int64_t s = i % v.S;
    int r = 0, a = 0, g = 0;
    const int st = site_eval(v, t, targets[t], s, r, a, g);
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double l0 = nan, l1 = nan, l2 = nan;
    if (st != 0) {
        if (v.tgt_counts) {
            const double *P = Ptab + (size_t)(r * C + a) * 3;
            l0 = lik_ibd0(f[s], P[0], P[1], P[2]);
            l1 = lik_ibd1(g, f[s], P[0], P[1], P[2]);
            l2 = P[g];
        } else {
            const double *L = lik7 + s * 7;
            l0 = L[0];
            l1 = L[1 + g];
            l2 = L[4 + g];
        }
    }
    if (st_out) st_out[i] = (uint8_t)st;
    if (lik_out) {
        lik_out[i * 3 + 0] = l0;
        lik_out[i * 3 + 1] = l1;
        lik_out[i * 3 + 2] = l2;
    }
}

// ---------------------------------------------------------------------------------------------
// K_LD_GENERAL: the --LD background loop (src/ibdgem.c:673-721) in log space, one CTA per
// (window, target, background block).  Each thread owns LD_PER background individuals and keeps
// their five running log-products (the chain P[r0+r1] and the four pseudo-diploid pairings
// P[a_i+r_j]) in registers; the window's informative sites are compacted into shared memory
// LD_THREADS candidates at a time.  The CTA then reduces its individuals to partial
// (max, sum-exp) pairs; exclusion of the target / pileup individual is by omission
// (src/ibdgem.c:714).  Handles every mode: per-target windows (-v), per-target counts (-D),
// arbitrary background lists and class tables.
constexpr int LD_THREADS = 256;
constexpr int LD_PER = 2;

struct LdPartial {
    double m0, s0, m1, s1;
};

__global__ void __launch_bounds__(LD_THREADS)
ld_general_kernel(SiteView v, WindowMapView m, const int32_t *__restrict__ targets,
                  const int32_t *__restrict__ bg, int n_bg, int pu_idx,
                  const double *__restrict__ lnPtab, int C, int outW, int nz,
                  LdPartial *__restrict__ part /*[T][outW][nz]*/) {
    const int w = blockIdx.x, t = blockIdx.y, z = blockIdx.z;
    const int row = (m.rows == 1) ? 0 : t;
    if (w >= m.nwin[row] || w >= m.maxW || w >= outW) return;
    const int indiv = targets[t];
    const int64_t s0 = m.wfirst[(int64_t)row * m.maxW + w], s1 = m.wlast[(int64_t)row * m.maxW + w];

    __shared__ double sl[LD_THREADS][3];
    __shared__ int64_t ssite[LD_THREADS];
    __shared__ uint8_t sa[LD_THREADS];
    __shared__ int wcount[LD_THREADS / 32];
    __shared__ double red[LD_THREADS / 32];

    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int b[LD_PER];
    bool valid[LD_PER];
    double acc[LD_PER][5];
#pragma unroll
    for (int p = 0; p < LD_PER; p++) {
        const int n = (z * LD_PER + p) * LD_THREADS + threadIdx.x;
        b[p] = (n < n_bg) ? bg[n] : -1;
        valid[p] = (n < n_bg) && b[p] != indiv && b[p] != pu_idx;
        if (!valid[p]) b[p] = 0;
#pragma unroll
        for (int q = 0; q < 5; q++) acc[p][q] = 0.0;
    }

    for (int64_t sb = s0; sb <= s1; sb += LD_THREADS) {
        // compact the informative sites of this candidate batch into shared memory, in order
        const int64_t s = sb + threadIdx.x;
        int r = 0, a = 0, g = 0;
        const bool inf = (s <= s1) && site_eval(v, t, indiv, s, r, a, g) == 1;
        const uint32_t bal = __ballot_sync(0xffffffffu, inf);
        if (lane == 0) wcount[wid] = __popc(bal);
        __syncthreads();
        int off = 0, cnt = 0;
        for (int k = 0; k < LD_THREADS / 32; k++) {
            if (k < wid) off += wcount[k];
            cnt += wcount[k];
        }
        if (inf) {
            const int j = off + __popc(bal & ((1u << lane) - 1u));
            const double *L = lnPtab + (size_t)(r * C + a) * 3;
            sl[j][0] = L[0];
            sl[j][1] = L[1];
            sl[j][2] = L[2];
            ssite[j] = s;
            sa[j] = (uint8_t)hap_pair(v.bits + s * v.Wh, indiv);
        }
        __syncthreads();
        for (int j = 0; j < cnt; j++) {
            const double l0 = sl[j][0], l1 = sl[j][1], l2 = sl[j][2];
            const uint32_t ta = sa[j];
            const double u0lo = (ta & 1u) ? l1 : l0, u0hi = (ta & 1u) ? l2 : l1;
            const double u1lo = (ta & 2u) ? l1 : l0, u1hi = (ta & 2u) ? l2 : l1;
            const uint32_t *rowp = v.bits + ssite[j] * v.Wh;
#pragma unroll
            for (int p = 0; p < LD_PER; p++) {
                const uint32_t pr = hap_pair(rowp, b[p]);
                const bool r0 = pr & 1u, r1 = pr & 2u;
                const int gg = (int)r0 + (int)r1;
                acc[p][0] += (gg == 0) ? l0 : (gg == 1 ? l1 : l2);
                acc[p][1] += r0 ? u0hi : u0lo;
                acc[p][2] += r1 ? u0hi : u0lo;
                acc[p][3] += r0 ? u1hi : u1lo;
                acc[p][4] += r1 ? u1hi : u1lo;
            }
        }
        __syncthreads();
    }

    // block log-sum-exp of the chain (IBD0) and of the 4 pairings (IBD1)
    const double NEG = -INFINITY;
    double m0 = NEG, m1 = NEG;
#pragma unroll
    for (int p = 0; p < LD_PER; p++)
        if (valid[p]) {
            m0 = fmax(m0, acc[p][0]);
            m1 = fmax(m1, fmax(fmax(acc[p][1], acc[p][2]), fmax(acc[p][3], acc[p][4])));
        }
    auto block_max = [&](double x) {
        x = warp_max_d(x);
        __syncthreads();
        if (lane == 0) red[wid] = x;
        __syncthreads();
        double y = red[0];
        for (int k = 1; k < LD_THREADS / 32; k++) y = fmax(y, red[k]);
        return y;
    };
    auto block_sum = [&](double x) {
        x = warp_sum_d(x);
        __syncthreads();
        if (lane == 0) red[wid] = x;
        __syncthreads();
        double y = 0;
        for (int k = 0; k < LD_THREADS / 32; k++) y += red[k];
        return y;
    };
    m0 = block_max(m0);
    m1 = block_max(m1);
    double e0 = 0, e1 = 0;
#pragma unroll
    for (int p = 0; p < LD_PER; p++)
        if (valid[p]) {
            e0 += exp(acc[p][0] - m0);
            e1 += exp(acc[p][1] - m1) + exp(acc[p][2] - m1) + exp(acc[p][3] - m1) + exp(acc[p][4] - m1);
        }
    e0 = block_sum(e0);
    e1 = block_sum(e1);
    if (threadIdx.x == 0) {
        LdPartial o;
        o.m0 = m0; o.s0 = e0; o.m1 = m1; o.s1 = e1;
        part[((int64_t)t * outW + w) * nz + z] = o;
    }
}

// K_LD_FINALIZE: merge the background-block partials and apply the divisors of
// src/ibdgem.c:751-752 (n_refpanel, 4*n_refpanel) in log space.
__global__ void ld_finalize_kernel(const LdPartial *__restrict__ part, int nz, WindowMapView m, int T,
                                   int outW, const int32_t *__restrict__ nrefpanel,
                                   double *__restrict__ wll) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * outW) return;
    const int t = (int)(i / outW), w = (int)(i % outW);
    const int row = (m.rows == 1) ? 0 : t;
    if (w >= m.nwin[row]) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const int nr = nrefpanel[t];
    if (nr <= 0) {  // 0/0 in the reference -> "-nan" (SURVEY.md §8a L2)
        wll[i * 3 + 0] = nan;
        wll[i * 3 + 1] = nan;
        return;
    }
    double M0 = -INFINITY, M1 = -INFINITY;
    for (int z = 0; z < nz; z++) {
        M0 = fmax(M0, part[i * nz + z].m0);
        M1 = fmax(M1, part[i * nz + z].m1);
    }
    double S0 = 0, S1 = 0;
    for (int z = 0; z < nz; z++) {
        const LdPartial p = part[i * nz + z];
        if (p.s0 > 0) S0 += p.s0 * exp(p.m0 - M0);
        if (p.s1 > 0) S1 += p.s1 * exp(p.m1 - M1);
    }
    wll[i * 3 + 0] = M0 + log(S0) - log((double)nr);
    wll[i * 3 + 1] = M1 + log(S1) - log(4.0 * (double)nr);
}

int wait_panel_upto(ibdgem_engine *e, int64_t s_end) {
    while (e->chunks_waited < (int)e->chunk_end.size() &&
           (e->chunks_waited == 0 || e->chunk_end[(size_t)e->chunks_waited - 1] < s_end)) {
        IBD_CUDA(cudaStreamWaitEvent(e->stream, e->chunk_ev[(size_t)e->chunks_waited], 0));
        e->chunks_waited++;
    }
    if (e->chunk_end.empty() || e->chunk_end.back() < s_end) {
        set_error("[::] ERROR: panel rows up to %lld are needed but only %lld were declared ready "
                  "(ibdgem_engine_panel_rows_ready).", (long long)s_end, (long long)(e->chunk_end.empty() ? 0 : e->chunk_end.back()));
        return 1;
    }
    return 0;
}

int ensure_table(ibdgem_engine *e, int64_t s_end) {
    if (wait_panel_upto(e, s_end)) return 1;
    if (e->table_upto >= s_end) return 0;
    {
        LaunchScope ls(e, K_SITE_TABLE);
        const int64_t n = s_end - e->table_upto;
        site_table_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(
            e->table_upto, s_end, e->N, e->Wh, e->d_bits, e->d_hostkeep, e->d_nref, e->d_nalt, e->d_afuser, e->d_P, e->C,
            e->prm.min_af, e->prm.max_af, (int)e->prm.max_cov, e->d_f, e->d_keep, e->d_status, e->d_lik7, e->d_lnlik7, e->d_lnP);
    }
    IBD_CUDA(cudaGetLastError());
    e->table_upto = s_end;
    return 0;
}

void window_shard_bounds(const ibdgem_engine *e, int32_t *w_begin, int32_t *w_end, int64_t *s_begin, int64_t *s_end) {
    const int64_t nW = e->nW_shared;
    const int32_t wb = (int32_t)(nW * e->shard_index / e->shard_count), we = (int32_t)(nW * (e->shard_index + 1) / e->shard_count);
    if (w_begin) *w_begin = wb;
    if (w_end) *w_end = we;
    // rows between two windows (uninformative sites) go with the later shard; the last shard runs to the end
    if (s_begin) *s_begin = wb > 0 && wb <= (int32_t)e->h_wlast.size() ? e->h_wlast[(size_t)wb - 1] + 1 : 0;
    if (s_end) *s_end = (e->shard_index + 1 >= e->shard_count || we <= 0 || we > (int32_t)e->h_wlast.size()) ? e->S : e->h_wlast[(size_t)we - 1] + 1;
}

}  // namespace ibdgem

using namespace ibdgem;

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char *ibdgem_last_error(void) { return g_err; }
int ibdgem_abi_version(void) { return IBDGEM_B200_ABI_VERSION; }

// M1 — nCk by the reference's recursion (src/ibd-math.c:5-10), unrolled deepest level first.
static unsigned long host_binom(unsigned int n, unsigned int k) {
    unsigned long v = 1;
    const unsigned int base = n - k;
    for (unsigned int j = 1; j <= k; j++) v = ((unsigned int)(base + j) * v) / j;
    return v;
}

// M2 — P(D|G) for one class (src/ibd-math.c:46-81), libm pow, (coef * p1) * p2.
// volatile keeps gcc from folding or contracting the double operations.
static void host_pdg(double eps, unsigned r, unsigned a, double out[3]) {
    if (r == 0 && a == 0) {
        out[0] = out[1] = out[2] = 1.0;
        return;
    }
    volatile double coef = (double)host_binom(r + a, r);
    volatile double p0 = coef * pow(1 - eps, (double)r);
    p0 = p0 * pow(eps, (double)a);
    volatile double p1 = coef * pow(0.5, (double)r);
    p1 = p1 * pow(0.5, (double)a);
    volatile double p2 = coef * pow(1 - eps, (double)a);
    p2 = p2 * pow(eps, (double)r);
    out[0] = p0 == 0.0 ? DBL_MIN : (double)p0;
    out[1] = p1 == 0.0 ? DBL_MIN : (double)p1;
    out[2] = p2 == 0.0 ? DBL_MIN : (double)p2;
}

int ibdgem_engine_create(const ibdgem_params *params, ibdgem_engine **out) {
    if (!params || !out) {
        set_error("[::] ERROR in ibdgem_engine_create(): NULL argument.");
        return 1;
    }
    *out = nullptr;
    if (params->max_cov < 1 || params->max_cov > IBDGEM_MAX_COV_LIMIT) {
        set_error("[::] ERROR: Invalid maximum estimated coverage (-M) of %u (must be 1..%d).",
                  params->max_cov, IBDGEM_MAX_COV_LIMIT);
        return 1;
    }
    if (params->window_size < 2) {
        set_error("[::] ERROR: Invalid window size (-w) of %d (must be >= 2).", params->window_size);
        return 1;
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0) {
        set_error("[::] ERROR: no usable CUDA device (%s); the engine has no CPU fallback.",
                  ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
        return 1;
    }
    if (params->device < 0 || params->device >= ndev) {
        set_error("[::] ERROR: CUDA device %d out of range (0..%d).", params->device, ndev - 1);
        return 1;
    }
    IBD_CUDA(cudaSetDevice(params->device));
    ibdgem_engine *e = new ibdgem_engine();
    e->prm = *params;
    e->device = params->device;
    e->C = (int)params->max_cov + 1;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, e->device) == cudaSuccess) e->sm_count = prop.multiProcessorCount;

    const int C = e->C;
    e->h_P.assign((size_t)C * C * 3, 1.0);
    e->h_lnP.assign((size_t)C * C * 3, 0.0);
    for (int r = 0; r < C; r++)
        for (int a = 0; a + r < C; a++) {
            double P[3];
            host_pdg(params->epsilon, (unsigned)r, (unsigned)a, P);
            for (int g = 0; g < 3; g++) {
                e->h_P[((size_t)r * C + a) * 3 + g] = P[g];
                e->h_lnP[((size_t)r * C + a) * 3 + g] = (double)logl((long double)P[g]);
            }
        }
    // Depth-linearity of the table (DESIGN.md "tensor path"): with no DBL_MIN clamp,
    //   lnP1 - lnP0 = r*alpha + a*beta   and   lnP2 - 2 lnP1 + lnP0 = (r + a) * kappa
    // with alpha = ln(0.5/(1-eps)), beta = ln(0.5/eps), kappa = ln(4 eps (1-eps)).
    {
        const long double eps = params->epsilon;
        bool ok = eps > 0 && eps < 1;
        long double kap = 0, al = 0, be = 0;
        if (ok) {
            kap = logl(4 * eps * (1 - eps));
            al = logl(0.5L / (1 - eps));
            be = logl(0.5L / eps);
            for (int r = 0; r < C && ok; r++)
                for (int a = 0; a + r < C && ok; a++) {
                    const double *L = &e->h_lnP[((size_t)r * C + a) * 3];
                    const long double c = (long double)L[2] - 2 * (long double)L[1] + L[0];
                    const long double d = (long double)L[1] - L[0];
                    const long double tol = 1e-12L * (1 + fabsl((long double)L[0]) + fabsl((long double)L[2]));
                    if (fabsl(c - (r + a) * kap) > tol || fabsl(d - (r * al + a * be)) > tol) ok = false;
                }
        }
        e->depth_linear = ok;
        e->kappa = (double)kap;
        e->alpha = (double)al;
        e->beta = (double)be;
    }
    if (dev_alloc(e, (void **)&e->d_P, e->h_P.size() * 8) || dev_alloc(e, (void **)&e->d_lnP, e->h_lnP.size() * 8)) {
        delete e;
        return 1;
    }
    IBD_CUDA(cudaMemcpy(e->d_P, e->h_P.data(), e->h_P.size() * 8, cudaMemcpyHostToDevice));
    IBD_CUDA(cudaMemcpy(e->d_lnP, e->h_lnP.data(), e->h_lnP.size() * 8, cudaMemcpyHostToDevice));
    *out = e;
    return 0;
}

static void free_sites(ibdgem_engine *e) {
    dev_free(e, e->d_pos, (size_t)e->S * 8);
    dev_free(e, e->d_nref, (size_t)e->S);
    dev_free(e, e->d_nalt, (size_t)e->S);
    dev_free(e, e->d_hostkeep, (size_t)e->S);
    if (e->d_afuser) dev_free(e, e->d_afuser, (size_t)e->S * 8);
    e->d_pos = nullptr;
    e->d_nref = e->d_nalt = e->d_hostkeep = nullptr;
    e->d_afuser = nullptr;
    e->have_sites = false;
}
static void free_panel(ibdgem_engine *e, int64_t S) {
    if (e->d_bits && e->owns_bits) dev_free(e, e->d_bits, (size_t)S * e->Wh * 4);
    e->d_bits = nullptr;
    e->owns_bits = true;
    e->have_panel = false;
}
static void free_prepared(ibdgem_engine *e, int64_t S) {
    if (e->d_f) {
        dev_free(e, e->d_f, (size_t)S * 8);
        dev_free(e, e->d_keep, (size_t)S);
        dev_free(e, e->d_status, (size_t)S);
        dev_free(e, e->d_lik7, (size_t)S * 56);
        dev_free(e, e->d_lnlik7, (size_t)S * 56);
        dev_free(e, e->d_rank, (size_t)S * 4);
    }
    if (e->d_wfirst) {
        const size_t cap = (size_t)(S / std::max(e->prm.window_size, 1) + 2) * 8;
        dev_free(e, e->d_wfirst, cap);
        dev_free(e, e->d_wlast, cap);
        dev_free(e, e->d_nwin_shared, 4);
        dev_free(e, e->d_ktot_shared, 8);
    }
    e->d_f = e->d_lik7 = e->d_lnlik7 = nullptr;
    e->d_keep = e->d_status = nullptr;
    e->d_rank = nullptr;
    e->d_wfirst = e->d_wlast = nullptr;
    e->d_nwin_shared = nullptr;
    e->d_ktot_shared = nullptr;
    e->prepared = false;
    ld_tensor_release(e);
    ld_vtensor_release(e);
}

int ibdgem_engine_destroy(ibdgem_engine *e) {
    if (!e) return 0;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    resolve_timers(e);
    const int64_t S = e->S;
    free_prepared(e, S);
    free_panel(e, S);
    if (e->have_sites) free_sites(e);
    dev_free(e, e->d_P, e->h_P.size() * 8);
    dev_free(e, e->d_lnP, e->h_lnP.size() * 8);
    dev_free(e, e->d_shared_cnt, (size_t)(e->C + 3) * 8);
    for (auto *b : e->scratch)
        if (b) {
            if (b->p) cudaFree(b->p);
            delete b;
        }
    for (auto ev : e->event_pool) cudaEventDestroy(ev);
    for (auto ev : e->chunk_ev) cudaEventDestroy(ev);
    if (e->ev_order) cudaEventDestroy(e->ev_order);
    if (e->ev_book) cudaEventDestroy(e->ev_book);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    for (auto ev : e->range_ev) cudaEventDestroy(ev);
    if (e->d2h_stream) cudaStreamDestroy(e->d2h_stream);
    if (e->h_pin) cudaFreeHost(e->h_pin);
    delete e;
    return 0;
}

int ibdgem_engine_set_stream(ibdgem_engine *e, void *cuda_stream) {
    if (!e) return 1;
    e->stream = (cudaStream_t)cuda_stream;
    return 0;
}

int ibdgem_engine_upload_sites(ibdgem_engine *e, int64_t n_sites, const uint64_t *pos,
                               const uint8_t *n_ref, const uint8_t *n_alt, const uint8_t *host_keep,
                               const double *af_user) {
    if (!e || n_sites <= 0 || !pos || !n_ref || !n_alt || !host_keep) {
        set_error("[::] ERROR in ibdgem_engine_upload_sites(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    if (!e->timeline_path) e->timeline_path = getenv("IBDGEM_TIMELINE");
    if (e->timeline_path && e->timing) {
        if (!e->ev_t0) {
            IBD_CUDA(cudaEventCreate(&e->ev_t0));
            IBD_CUDA(cudaEventCreate(&e->ev_wll));
            IBD_CUDA(cudaEventCreate(&e->ev_bookdone));
        }
        IBD_CUDA(cudaEventRecord(e->ev_t0, e->stream));
        e->t0_set = true;
    }
    if (e->have_panel && e->S != n_sites) {
        set_error("[::] ERROR: site count %lld does not match the uploaded panel (%lld rows).",
                  (long long)n_sites, (long long)e->S);
        return 1;
    }
    if (e->have_sites && (e->S != n_sites || (af_user != nullptr) != (e->d_afuser != nullptr))) {
        const int64_t S_old = e->S;
        free_prepared(e, S_old);
        free_sites(e);
    }
    if (!e->have_sites) {
        if (!e->have_panel) e->S = n_sites;
        if (dev_alloc(e, (void **)&e->d_pos, (size_t)n_sites * 8) || dev_alloc(e, (void **)&e->d_nref, (size_t)n_sites) ||
            dev_alloc(e, (void **)&e->d_nalt, (size_t)n_sites) || dev_alloc(e, (void **)&e->d_hostkeep, (size_t)n_sites))
            return 1;
        if (af_user && dev_alloc(e, (void **)&e->d_afuser, (size_t)n_sites * 8)) return 1;
    }
    IBD_CUDA(cudaMemcpyAsync(e->d_pos, pos, (size_t)n_sites * 8, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(e->d_nref, n_ref, (size_t)n_sites, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(e->d_nalt, n_alt, (size_t)n_sites, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(e->d_hostkeep, host_keep, (size_t)n_sites, cudaMemcpyHostToDevice, e->stream));
    if (af_user)
        IBD_CUDA(cudaMemcpyAsync(e->d_afuser, af_user, (size_t)n_sites * 8, cudaMemcpyHostToDevice, e->stream));
    e->have_sites = true;
    e->prepared = false;
    return 0;
}

int ibdgem_engine_upload_panel(ibdgem_engine *e, int64_t n_sites, int32_t n_indiv,
                               const uint32_t *bits, int64_t words_per_site) {
    if (!e || n_sites <= 0 || n_indiv <= 0 || !bits || words_per_site * 32 < 2 * (int64_t)n_indiv) {
        set_error("[::] ERROR in ibdgem_engine_upload_panel(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    if (e->have_sites && e->S != n_sites) {
        set_error("[::] ERROR: panel has %lld rows but %lld sites were uploaded.", (long long)n_sites,
                  (long long)e->S);
        return 1;
    }
    if (e->have_panel && (e->S != n_sites || e->Wh != words_per_site)) {
        free_prepared(e, e->S);
        free_panel(e, e->S);
    }
    if (e->have_panel && !e->owns_bits) free_panel(e, e->S);  // never copy into the caller's device buffer
    if (!e->have_panel) {
        e->S = n_sites;
        e->Wh = words_per_site;
        if (dev_alloc(e, (void **)&e->d_bits, (size_t)n_sites * words_per_site * 4)) return 1;
    }
    e->N = n_indiv;
    // chunked copy on the copy stream, ordered after whatever the engine stream still reads from d_bits
    if (!e->copy_stream) {
        IBD_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        IBD_CUDA(cudaEventCreateWithFlags(&e->ev_order, cudaEventDisableTiming));
    }
    // Equal chunks.  Scoring a chunk's windows takes less time than copying it (C3: 9.0 ms of scoring
    // against 11.6 ms of PCIe for the whole panel), so the GPU keeps up with the copy and the end-to-end
    // step is ~ copy + one chunk's scoring + its result copy.  Measured at C3 (bench.py e2e, ms):
    // 1 chunk 22.5, 5: 13.6, 8: 13.1, 12: 12.8, 16: 12.65, 20: 12.6, 24: 13.3, 32: 14.9, 64: 20.2 — past ~20 the
    // per-range launches (a dozen per range) cost more than the shorter tail saves.  Tapered sizes
    // (IBDGEM_PANEL_TAPER < 1) measured no better: the scoring rate is too close to the copy rate for
    // shrinking chunks to stay ahead.
    // read once (C++11 static initialisers are thread-safe: `ibdgem --gpus N` calls this from one host
    // thread per device)
    static const int want_chunks = [] {
        const char *sc = getenv("IBDGEM_PANEL_CHUNKS");
        return sc ? std::max(1, atoi(sc)) : PANEL_CHUNKS;
    }();
    static const double taper = [] {  // each chunk is `taper` times the size of the one before it
        const char *st = getenv("IBDGEM_PANEL_TAPER");
        const double t = st ? atof(st) : PANEL_TAPER;
        return (t > 0.1 && t <= 1.0) ? t : 1.0;
    }();
    const size_t panel_bytes = (size_t)n_sites * (size_t)words_per_site * 4;
    const int nchunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)want_chunks, panel_bytes / PANEL_CHUNK_MIN_BYTES));
    while ((int)e->chunk_ev.size() < nchunk) {
        cudaEvent_t ev;
        IBD_CUDA(cudaEventCreateWithFlags(&ev, e->t0_set ? cudaEventDefault : cudaEventDisableTiming));
        e->chunk_ev.push_back(ev);
    }
    IBD_CUDA(cudaEventRecord(e->ev_order, e->stream));
    IBD_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_order, 0));
    e->chunk_end.assign((size_t)nchunk, 0);
    double wsum = 0, wk = 1;
    for (int k = 0; k < nchunk; k++, wk *= taper) wsum += wk;
    int64_t s0 = 0;
    double acc = 0;
    wk = 1;
    for (int k = 0; k < nchunk; k++, wk *= taper) {
        acc += wk / wsum;
        const int64_t s1 = k + 1 == nchunk ? n_sites : std::min<int64_t>(n_sites, std::max<int64_t>(s0 + 1, (int64_t)(acc * (double)n_sites)));
        IBD_CUDA(cudaMemcpyAsync(e->d_bits + (size_t)s0 * words_per_site, bits + (size_t)s0 * words_per_site,
                                 (size_t)(s1 - s0) * words_per_site * 4, cudaMemcpyHostToDevice, e->copy_stream));
        IBD_CUDA(cudaEventRecord(e->chunk_ev[(size_t)k], e->copy_stream));
        e->chunk_end[(size_t)k] = s1;
        s0 = s1;
    }
    e->chunks_waited = 0;
    e->have_panel = true;
    e->prepared = false;
    e->table_from = e->table_upto = 0;
    ld_tensor_invalidate(e);
    ld_vtensor_invalidate(e);
    return 0;
}

int ibdgem_engine_set_panel_device(ibdgem_engine *e, int64_t n_sites, int32_t n_indiv, const uint32_t *d_bits,
                                   int64_t words_per_site) {
    if (!e || n_sites <= 0 || n_indiv <= 0 || !d_bits || words_per_site * 32 < 2 * (int64_t)n_indiv) {
        set_error("[::] ERROR in ibdgem_engine_set_panel_device(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, d_bits) != cudaSuccess || attr.type != cudaMemoryTypeDevice || attr.device != e->device) {
        cudaGetLastError();
        set_error("[::] ERROR in ibdgem_engine_set_panel_device(): d_bits is not device memory of GPU %d.", e->device);
        return 1;
    }
    if (e->have_sites && e->S != n_sites) {
        set_error("[::] ERROR: panel has %lld rows but %lld sites were uploaded.", (long long)n_sites, (long long)e->S);
        return 1;
    }
    // kernels of an earlier call may still read the old buffer
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    if (e->have_panel && (e->S != n_sites || e->Wh != words_per_site)) free_prepared(e, e->S);
    if (e->have_panel) free_panel(e, e->S);
    e->S = n_sites;
    e->Wh = words_per_site;
    e->N = n_indiv;
    e->d_bits = const_cast<uint32_t *>(d_bits);
    e->owns_bits = false;
    e->chunk_end.clear();
    e->chunks_waited = 0;
    e->have_panel = true;
    e->prepared = false;
    e->table_from = e->table_upto = 0;
    ld_tensor_invalidate(e);
    ld_vtensor_invalidate(e);
    return 0;
}

// The packed panel of `src` (another engine of this process, usually on another GPU) copied device to device over
// NVLink, chunk by chunk as src's own upload lands: one PCIe upload per node instead of one per engine.
int ibdgem_engine_clone_panel(ibdgem_engine *e, ibdgem_engine *src) {
    if (!e || !src || e == src || !src->have_panel) {
        set_error("[::] ERROR in ibdgem_engine_clone_panel(): the source engine has no panel.");
        return 1;
    }
    if (e->have_sites && e->S != src->S) {
        set_error("[::] ERROR: panel has %lld rows but %lld sites were uploaded.", (long long)src->S, (long long)e->S);
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    if (e->have_panel && (e->S != src->S || e->Wh != src->Wh || !e->owns_bits)) {
        free_prepared(e, e->S);
        free_panel(e, e->S);
    }
    if (!e->have_panel) {
        e->S = src->S;
        e->Wh = src->Wh;
        if (dev_alloc(e, (void **)&e->d_bits, (size_t)e->S * e->Wh * 4)) return 1;
    }
    e->N = src->N;
    if (!e->copy_stream) {
        IBD_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        IBD_CUDA(cudaEventCreateWithFlags(&e->ev_order, cudaEventDisableTiming));
    }
    if (e->device != src->device) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, e->device, src->device);
        if (can && cudaDeviceEnablePeerAccess(src->device, 0) == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
    }
    IBD_CUDA(cudaEventRecord(e->ev_order, e->stream));
    IBD_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_order, 0));
    // src's chunk layout: a caller-owned source panel (no chunks of its own) is taken as one piece, already complete
    const size_t nchunk = std::max<size_t>(1, src->chunk_end.size());
    while (e->chunk_ev.size() < nchunk) {
        cudaEvent_t ev;
        IBD_CUDA(cudaEventCreateWithFlags(&ev, e->t0_set ? cudaEventDefault : cudaEventDisableTiming));
        e->chunk_ev.push_back(ev);
    }
    e->chunk_end.assign(nchunk, 0);
    int64_t s0 = 0;
    for (size_t k = 0; k < nchunk; k++) {
        const int64_t s1 = src->chunk_end.empty() ? src->S : src->chunk_end[k];
        if (!src->chunk_end.empty()) IBD_CUDA(cudaStreamWaitEvent(e->copy_stream, src->chunk_ev[k], 0));
        IBD_CUDA(cudaMemcpyPeerAsync(e->d_bits + (size_t)s0 * e->Wh, e->device, src->d_bits + (size_t)s0 * e->Wh, src->device,
                                     (size_t)(s1 - s0) * e->Wh * 4, e->copy_stream));
        IBD_CUDA(cudaEventRecord(e->chunk_ev[k], e->copy_stream));
        e->chunk_end[k] = s1;
        s0 = s1;
    }
    e->chunks_waited = 0;
    e->have_panel = true;
    e->owns_bits = true;
    e->prepared = false;
    e->table_from = e->table_upto = 0;
    ld_tensor_invalidate(e);
    ld_vtensor_invalidate(e);
    return 0;
}

int ibdgem_engine_panel_rows_ready(ibdgem_engine *e, int64_t row_end, void *stream) {
    if (!e || !e->have_panel || e->owns_bits) {
        set_error("[::] ERROR in ibdgem_engine_panel_rows_ready(): no caller-owned device panel is set.");
        return 1;
    }
    if (row_end <= 0 || row_end > e->S || (!e->chunk_end.empty() && row_end < e->chunk_end.back())) {
        set_error("[::] ERROR in ibdgem_engine_panel_rows_ready(): row_end %lld out of order or range.", (long long)row_end);
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    const size_t k = e->chunk_end.size();
    while (e->chunk_ev.size() <= k) {
        cudaEvent_t ev;
        IBD_CUDA(cudaEventCreateWithFlags(&ev, e->t0_set ? cudaEventDefault : cudaEventDisableTiming));
        e->chunk_ev.push_back(ev);
    }
    IBD_CUDA(cudaEventRecord(e->chunk_ev[k], stream ? static_cast<cudaStream_t>(stream) : e->stream));
    e->chunk_end.push_back(row_end);
    return 0;
}

int ibdgem_engine_sync_uploads(ibdgem_engine *e) {
    if (!e) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    if (e->copy_stream) IBD_CUDA(cudaStreamSynchronize(e->copy_stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

static SiteView make_view(ibdgem_engine *e, const uint8_t *d_tgt_counts, int vflag) {
    SiteView v;
    v.keep = e->d_keep;
    v.nref = e->d_nref;
    v.nalt = e->d_nalt;
    v.bits = e->d_bits;
    v.Wh = e->Wh;
    v.S = e->S;
    v.tgt_counts = d_tgt_counts;
    v.vflag = vflag;
    return v;
}

// Builds a window map for `rows` rows (targets==nullptr -> one shared row).
extern "C++" {
namespace ibdgem {
int build_window_map(ibdgem_engine *e, const SiteView &v, const int32_t *d_targets, int rows,
                     int maxW, int64_t *d_wfirst, int64_t *d_wlast, int32_t *d_nwin,
                     int64_t *d_ktot, uint32_t *d_rank) {
    const int nb = (int)((e->S + SCAN_CHUNK - 1) / SCAN_CHUNK);
    uint32_t *d_cnt;
    if (scratch(e, SC_BLOCKCNT, (size_t)rows * nb * 4, (void **)&d_cnt)) return 1;
    // rows ride on gridDim.y (limit 65,535): slices of ROW_SLICE rows
    for (int r0 = 0; r0 < rows; r0 += ROW_SLICE) {
        const int rc = std::min(ROW_SLICE, rows - r0);
        SiteView vv = v;
        if (vv.tgt_counts) vv.tgt_counts += (size_t)r0 * e->S * 2;
        const int32_t *tg = d_targets ? d_targets + r0 : nullptr;
        uint32_t *cnt = d_cnt + (size_t)r0 * nb;
        {
            LaunchScope ls(e, K_SCAN_COUNT);
            scan_count_kernel<<<dim3(nb, rc), SCAN_THREADS, 0, e->stream>>>(vv, tg, cnt, nb);
        }
        {
            LaunchScope ls(e, K_SCAN_OFFSETS);
            scan_offsets_kernel<<<rc, 256, 0, e->stream>>>(cnt, nb, e->prm.window_size, d_ktot + r0, d_nwin + r0);
        }
        {
            LaunchScope ls(e, K_SCAN_RANK);
            scan_rank_kernel<<<dim3(nb, rc), SCAN_THREADS, 0, e->stream>>>(
                vv, tg, cnt, nb, e->prm.window_size, d_ktot + r0, d_wfirst + (size_t)r0 * maxW, d_wlast + (size_t)r0 * maxW, maxW,
                d_rank);
        }
    }
    IBD_CUDA(cudaGetLastError());
    return 0;
}
}  // namespace ibdgem
}  // extern "C++"

int ibdgem_engine_prepare(ibdgem_engine *e) {
    if (!e) return 1;
    if (e->prepared) return 0;
    if (!e->have_sites || !e->have_panel) {
        set_error("[::] ERROR in ibdgem_engine_prepare(): sites and panel must both be uploaded.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    const int64_t S = e->S;
    const int maxW = (int)(S / e->prm.window_size + 2);
    if (!e->d_f) {
        if (dev_alloc(e, (void **)&e->d_f, (size_t)S * 8) || dev_alloc(e, (void **)&e->d_keep, (size_t)S) ||
            dev_alloc(e, (void **)&e->d_status, (size_t)S) || dev_alloc(e, (void **)&e->d_lik7, (size_t)S * 56) ||
            dev_alloc(e, (void **)&e->d_lnlik7, (size_t)S * 56) || dev_alloc(e, (void **)&e->d_rank, (size_t)S * 4) ||
            dev_alloc(e, (void **)&e->d_wfirst, (size_t)maxW * 8) || dev_alloc(e, (void **)&e->d_wlast, (size_t)maxW * 8) ||
            dev_alloc(e, (void **)&e->d_nwin_shared, 4) || dev_alloc(e, (void **)&e->d_ktot_shared, 8))
            return 1;
    }
    e->table_from = e->table_upto = 0;
    // With no -A table and the default AF range the filter verdicts do not depend on the panel:
    // the window map is built from the site arrays at once, and the per-site table (which reads the
    // panel) is evaluated chunk by chunk as the rows arrive (ensure_table).
    e->lazy_table = !e->d_afuser && e->prm.min_af <= 0.0 && e->prm.max_af >= 1.0;
    e->shared_cnt_valid = false;
    if (e->lazy_table) {
        if (!e->d_shared_cnt && dev_alloc(e, (void **)&e->d_shared_cnt, (size_t)(e->C + 3) * 8)) return 1;
        IBD_CUDA(cudaMemsetAsync(e->d_shared_cnt, 0, (size_t)(e->C + 3) * 8, e->stream));
        LaunchScope ls(e, K_SITE_TABLE);
        const unsigned nblk = (unsigned)std::min<int64_t>((S + 255) / 256, (int64_t)e->sm_count * 8);
        site_status_kernel<<<nblk, 256, (size_t)(e->C + 3) * 4, e->stream>>>(S, e->d_hostkeep, e->d_nref, e->d_nalt, (int)e->prm.max_cov,
                                                                           e->d_keep, e->d_status, e->C, e->d_shared_cnt);
        e->shared_cnt_valid = true;
    } else if (ensure_table(e, S)) {
        return 1;
    }
    IBD_CUDA(cudaGetLastError());
    int32_t *d_nwin = e->d_nwin_shared;
    int64_t *d_ktot = e->d_ktot_shared;
    SiteView v = make_view(e, nullptr, 0);
    v.bits = nullptr;  // the shared map (vflag = 0, no per-target counts) never looks at genotypes
    if (build_window_map(e, v, nullptr, 1, maxW, e->d_wfirst, e->d_wlast, d_nwin, d_ktot, e->d_rank)) return 1;
    // window count, kept-site total and the last site of every window in one round trip through pinned
    // memory (the map has at most maxW windows)
    int64_t *h_map;
    if (pinned_stage(e, (size_t)(maxW + 2) * 8, (void **)&h_map)) return 1;
    IBD_CUDA(cudaMemcpyAsync(h_map, d_nwin, 4, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaMemcpyAsync(h_map + 1, d_ktot, 8, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaMemcpyAsync(h_map + 2, e->d_wlast, (size_t)maxW * 8, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    const int32_t nwin = *reinterpret_cast<const int32_t *>(h_map);
    const int64_t ktot = h_map[1];
    e->nW_shared = nwin;
    e->K_shared = ktot;
    e->h_wlast.assign(h_map + 2, h_map + 2 + std::max(nwin, 0));
    e->table_from = 0;
    if (e->shard_count > 1 && e->lazy_table) {  // a window shard evaluates the per-site table of its own rows only
        int64_t sb = 0;
        window_shard_bounds(e, nullptr, nullptr, &sb, nullptr);
        e->table_from = e->table_upto = sb;
    }
    e->prepared = true;
    ld_tensor_invalidate(e);
    ld_vtensor_invalidate(e);
    settle_timers(e);
    return 0;
}

int ibdgem_engine_invalidate(ibdgem_engine *e) {
    if (!e) return 1;
    e->prepared = false;
    e->table_from = e->table_upto = 0;
    ld_tensor_invalidate(e);
    ld_vtensor_invalidate(e);
    return 0;
}

int ibdgem_engine_get_site_table(ibdgem_engine *e, double *f, uint8_t *status, double *lik7) {
    if (!e) return 1;
    if (ibdgem_engine_prepare(e)) return 1;
    if (e->table_from > 0) {  // a window shard skipped the rows before its own: the whole table is wanted now
        e->table_from = 0;
        e->table_from = e->table_upto = 0;
    }
    if (ensure_table(e, e->S)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    if (f) IBD_CUDA(cudaMemcpyAsync(f, e->d_f, (size_t)e->S * 8, cudaMemcpyDeviceToHost, e->stream));
    if (status) IBD_CUDA(cudaMemcpyAsync(status, e->d_status, (size_t)e->S, cudaMemcpyDeviceToHost, e->stream));
    if (lik7) IBD_CUDA(cudaMemcpyAsync(lik7, e->d_lik7, (size_t)e->S * 56, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

static int score_common(ibdgem_engine *e, int32_t T, const int32_t *targets, int32_t n_bg,
                        const int32_t *bg, int32_t pu_idx, const uint8_t *tgt_counts,
                        ibdgem_scores *out, bool ld) {
    if (!e || T <= 0 || !targets || !out || (ld && (n_bg < 0 || (n_bg > 0 && !bg)))) {
        set_error("[::] ERROR in ibdgem_engine_score_%s(): bad arguments.", ld ? "ld" : "nonld");
        return 1;
    }
    if (ibdgem_engine_prepare(e)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    for (int t = 0; t < T; t++)
        if (targets[t] < 0 || targets[t] >= e->N) {
            set_error("[::] ERROR: target ordinal %d out of range (panel has %d individuals).", targets[t], e->N);
            return 1;
        }
    for (int n = 0; ld && n < n_bg; n++)
        if (bg[n] < 0 || bg[n] >= e->N) {
            set_error("[::] ERROR: background ordinal %d out of range (panel has %d individuals).", bg[n], e->N);
            return 1;
        }
    const int64_t S = e->S;
    const int C = e->C;
    const int vflag = e->prm.variable_sites_only ? 1 : 0;
    const bool shared = !vflag && !tgt_counts;
    const int mapW = shared ? std::max(e->nW_shared, 1) : (int)(S / e->prm.window_size + 2);
    const bool want_windows = out->n_windows || out->w_start || out->w_end || out->w_nsites || out->w_loglik ||
                              out->w_loglik_device || out->w_lik_linear;
    const int outW = want_windows ? out->max_windows : mapW;
    if (want_windows && outW <= 0) {
        set_error("[::] ERROR: ibdgem_scores.max_windows must be positive.");
        return 1;
    }
    if (shared && want_windows && e->nW_shared > outW) {
        set_error("[::] ERROR: %d windows do not fit max_windows = %d.", e->nW_shared, outW);
        return 1;
    }

    int32_t *d_targets;
    if (scratch(e, SC_TARGETS, (size_t)T * 4, (void **)&d_targets)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_targets, targets, (size_t)T * 4, cudaMemcpyHostToDevice, e->stream));
    uint8_t *d_tc = nullptr;
    if (tgt_counts) {
        if (scratch(e, SC_TGT_COUNTS, (size_t)T * S * 2, (void **)&d_tc)) return 1;
        IBD_CUDA(cudaMemcpyAsync(d_tc, tgt_counts, (size_t)T * S * 2, cudaMemcpyHostToDevice, e->stream));
    }
    SiteView v = make_view(e, d_tc, vflag);

    // window map
    bool vtensor = false;
    WindowMapView m;
    int32_t *d_nwin;
    int64_t *d_ktot;
    if (shared) {
        d_nwin = e->d_nwin_shared;
        m.wfirst = e->d_wfirst;
        m.wlast = e->d_wlast;
        m.nwin = d_nwin;
        m.rows = 1;
        m.maxW = (int)(S / e->prm.window_size + 2);
    } else if (ld && !e->force_general && ld_vtensor_eligible(e, T, n_bg)) {
        vtensor = true;  // the per-target-window tensor path builds its own window map (in rank space for -v)
        d_nwin = nullptr;
        m.wfirst = m.wlast = nullptr;
        m.nwin = nullptr;
        m.rows = T;
        m.maxW = mapW;
    } else {
        int64_t *d_wf, *d_wl;
        if (scratch(e, SC_WFIRST, (size_t)T * mapW * 8, (void **)&d_wf) ||
            scratch(e, SC_WLAST, (size_t)T * mapW * 8, (void **)&d_wl) ||
            scratch(e, SC_NWIN, (size_t)std::max(T, 1) * 4, (void **)&d_nwin) ||
            scratch(e, SC_KTOT, (size_t)std::max(T, 1) * 8, (void **)&d_ktot))
            return 1;
        // -v ranks sites by the target's genotype, i.e. reads panel rows: the engine stream must depend on
        // every panel chunk (and the per-site table) BEFORE the map is built, not only before the scoring
        // kernels — a lazily prepared engine has so far only looked at the site arrays
        if (ensure_table(e, S)) return 1;
        if (build_window_map(e, v, d_targets, T, mapW, d_wf, d_wl, d_nwin, d_ktot, nullptr)) return 1;
        m.wfirst = d_wf;
        m.wlast = d_wl;
        m.nwin = d_nwin;
        m.rows = T;
        m.maxW = mapW;
    }

    // non-LD window sums (LIBD2 of --LD runs is the non-LD product too, src/ibdgem.c:752)
    double *d_wll;
    int32_t *d_wn, *d_nwout;
    uint64_t *d_ws, *d_we;
    const size_t nWT = (size_t)T * outW;
    if (scratch(e, SC_WLL, nWT * 24, (void **)&d_wll) || scratch(e, SC_WN, nWT * 4 + (size_t)T * 4, (void **)&d_wn) ||
        scratch(e, SC_WS, nWT * 8, (void **)&d_ws) || scratch(e, SC_WE, nWT * 8, (void **)&d_we))
        return 1;
    d_nwout = d_wn + nWT;
    {
        LaunchScope ls(e, K_FILL);
        fill_nan_kernel<<<(unsigned)std::min<int64_t>((int64_t)(nWT * 3 + 255) / 256, 4096), 256, 0, e->stream>>>(d_wll, (int64_t)nWT * 3);
    }
    IBD_CUDA(cudaMemsetAsync(d_wn, 0, nWT * 4 + (size_t)T * 4, e->stream));
    IBD_CUDA(cudaMemsetAsync(d_ws, 0, nWT * 8, e->stream));
    IBD_CUDA(cudaMemsetAsync(d_we, 0, nWT * 8, e->stream));
    const bool tensor = ld && !e->force_general && shared && ld_tensor_eligible(e, T, n_bg, tgt_counts);
    e->book_ready = false;
    if ((tensor || vtensor) && !e->copy_stream) {  // (a panel set in device memory never went through upload_panel)
        IBD_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        IBD_CUDA(cudaEventCreateWithFlags(&e->ev_order, cudaEventDisableTiming));
    }
    if ((tensor || vtensor) && !e->ev_book) IBD_CUDA(cudaEventCreateWithFlags(&e->ev_book, cudaEventDisableTiming));
    // everything but the tensor path reads the per-site table and the whole panel up front; the
    // tensor path asks for them window range by window range (upload / scoring overlap)
    if (!tensor) {
        if (e->shard_count > 1) {
            set_error("[::] ERROR: a window shard (ibdgem_engine_set_window_shard) needs the shared-window tensor --LD path; "
                      "shard the target list instead for non-LD, -v and -D runs.");
            return 1;
        }
        if (ensure_table(e, S)) return 1;
    }
    e->wll_streamed = false;
    e->wll_dev_streamed = false;
    e->h_wll_out = out->w_loglik;
    e->d_wll_out_device = static_cast<double *>(out->w_loglik_device);
    if (vtensor) {
        const int rc = ld_vtensor_score(e, T, targets, d_targets, n_bg, bg, pu_idx, d_tc, outW, d_wll, d_wn, d_ws, d_we, d_nwout);
        if (rc == 1) return 1;
        if (rc == 2) {  // not taken after all (e.g. every background member excluded): the general path, with its own map
            vtensor = false;
            int64_t *d_wf, *d_wl;
            if (scratch(e, SC_WFIRST, (size_t)T * mapW * 8, (void **)&d_wf) ||
                scratch(e, SC_WLAST, (size_t)T * mapW * 8, (void **)&d_wl) ||
                scratch(e, SC_NWIN, (size_t)std::max(T, 1) * 4, (void **)&d_nwin) ||
                scratch(e, SC_KTOT, (size_t)std::max(T, 1) * 8, (void **)&d_ktot))
                return 1;
            if (build_window_map(e, v, d_targets, T, mapW, d_wf, d_wl, d_nwin, d_ktot, nullptr)) return 1;
            m.wfirst = d_wf;
            m.wlast = d_wl;
            m.nwin = d_nwin;
        } else {
            e->last_ld_path = 2;
        }
    }
    if (vtensor) {
        // done: window bookkeeping, LIBD0, LIBD1 and LIBD2 of every target are in place
    } else if (tensor) {
        // tensor path: fills window bookkeeping, LIBD0, LIBD1 and LIBD2 of every target
        if (ld_tensor_score(e, T, targets, d_targets, n_bg, bg, pu_idx, outW, d_wll, d_wn, d_ws, d_we, d_nwout)) return 1;
        e->last_ld_path = 1;
    } else {
        {
            LaunchScope ls(e, K_WINDOW_NONLD);
            if (shared) {
                // IBDGEM_NONLD_BATCH: 8 / 16 / 32 genotype loads in flight per thread (A/B: measured 0.154 / 0.181 / 0.242 ms at C2 — more loads in flight cost more in resident CTAs than they save)
                static const int batch = [] { const char *sb = getenv("IBDGEM_NONLD_BATCH"); return sb ? atoi(sb) : 8; }();
                const dim3 grid((unsigned)std::max(e->nW_shared, 1), (unsigned)((T + 127) / 128));
                auto kern = batch >= 32 ? window_nonld_shared_kernel<32> : (batch >= 16 ? window_nonld_shared_kernel<16> : window_nonld_shared_kernel<8>);
                kern<<<grid, 128, 0, e->stream>>>(v, m, d_targets, T, e->d_pos, e->d_status, e->d_lnlik7, outW, d_wll, d_wn, d_ws, d_we, d_nwout);
            } else {
                const int64_t warps = (int64_t)nWT;
                window_nonld_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, e->stream>>>(
                    v, m, d_targets, T, e->d_pos, e->d_f, e->d_lnlik7, e->d_P, C, outW, d_wll, d_wn, d_ws, d_we, d_nwout);
            }
        }
        IBD_CUDA(cudaGetLastError());
    }

    if (ld && !tensor && !vtensor) {
        std::vector<int32_t> h_nref(T);
        for (int t = 0; t < T; t++) {
            int c = 0;
            for (int n = 0; n < n_bg; n++)
                if (bg[n] != targets[t] && bg[n] != pu_idx) c++;
            h_nref[t] = c;
        }
        {
            int32_t *d_bg, *d_nrp;
            LdPartial *d_part;
            const int nz = std::max(1, (n_bg + LD_THREADS * LD_PER - 1) / (LD_THREADS * LD_PER));
            if (scratch(e, SC_BG, (size_t)std::max(n_bg, 1) * 4, (void **)&d_bg) ||
                scratch(e, SC_NREFPANEL, (size_t)T * 4, (void **)&d_nrp) ||
                scratch(e, SC_LD_PART, nWT * nz * sizeof(LdPartial), (void **)&d_part))
                return 1;
            if (n_bg > 0) IBD_CUDA(cudaMemcpyAsync(d_bg, bg, (size_t)n_bg * 4, cudaMemcpyHostToDevice, e->stream));
            IBD_CUDA(cudaMemcpyAsync(d_nrp, h_nref.data(), (size_t)T * 4, cudaMemcpyHostToDevice, e->stream));
            // grid.y/z are limited to 65535: chunk the targets
            for (int t0 = 0; t0 < T; t0 += 32768) {
                const int tc = std::min(32768, T - t0);
                SiteView vv = v;
                if (vv.tgt_counts) vv.tgt_counts += (size_t)t0 * S * 2;
                WindowMapView mm = m;
                if (mm.rows != 1) {
                    mm.wfirst += (size_t)t0 * m.maxW;
                    mm.wlast += (size_t)t0 * m.maxW;
                    mm.nwin += t0;
                }
                LaunchScope ls(e, K_LD_GENERAL);
                ld_general_kernel<<<dim3(outW, tc, nz), LD_THREADS, 0, e->stream>>>(
                    vv, mm, d_targets + t0, d_bg, n_bg, pu_idx, e->d_lnP, C, outW, nz, d_part + (size_t)t0 * outW * nz);
            }
            {
                LaunchScope ls(e, K_LD_FINALIZE);
                ld_finalize_kernel<<<(unsigned)((nWT + 255) / 256), 256, 0, e->stream>>>(d_part, nz, m, T, outW, d_nrp, d_wll);
            }
            IBD_CUDA(cudaGetLastError());
            e->last_ld_path = 0;
        }
    }

    if (e->shard_count == 1 && ensure_table(e, S)) return 1;  // no-op unless the tensor path left a tail
    // the reference's own linear window products, on request (not for --LD with per-target windows: that path keeps its
    // window map in rank space)
    double *d_wlin = nullptr;
    if (out->w_lik_linear && e->shard_count == 1) {
        if (scratch(e, SC_WLIN, nWT * 24, (void **)&d_wlin)) return 1;
        {
            LaunchScope ls(e, K_FILL);
            fill_nan_kernel<<<(unsigned)std::min<int64_t>((int64_t)(nWT * 3 + 255) / 256, 4096), 256, 0, e->stream>>>(d_wlin, (int64_t)nWT * 3);
        }
        if (!vtensor) {
            LaunchScope ls(e, K_WINDOW_LINEAR);
            window_linear_kernel<<<(unsigned)((nWT + 127) / 128), 128, 0, e->stream>>>(v, m, d_targets, T, e->d_f, e->d_lik7, e->d_P, C, outW, d_wlin);
        }
        IBD_CUDA(cudaGetLastError());
    }
    // counters
    const bool want_counters = out->processed || out->skipped || out->final_total_cov || out->final_dist;
    unsigned long long *d_cnt = nullptr;
    const int crow = C + 3;
    const int crows = shared ? 1 : T;
    if (want_counters && shared && e->shared_cnt_valid) {
        d_cnt = e->d_shared_cnt;  // counted by site_status_kernel in prepare()
    } else if (want_counters) {
        if (scratch(e, SC_COUNTERS, (size_t)crows * crow * 8, (void **)&d_cnt)) return 1;
        IBD_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)crows * crow * 8, e->stream));
        LaunchScope ls(e, K_COUNTERS);
        for (int r0 = 0; r0 < crows; r0 += ROW_SLICE) {
            const int rc = std::min(ROW_SLICE, crows - r0);
            SiteView vv = v;
            if (vv.tgt_counts) vv.tgt_counts += (size_t)r0 * S * 2;
            counters_kernel<<<dim3((unsigned)((S + COUNTERS_CHUNK - 1) / COUNTERS_CHUNK), rc), 256, (size_t)crow * 8, e->stream>>>(
                vv, shared ? nullptr : d_targets + r0, C, d_cnt + (size_t)r0 * crow);
        }
    }
    // expanded per-site outputs
    uint8_t *d_st = nullptr;
    double *d_sl = nullptr;
    if (out->site_status || out->site_lik) {
        if (out->site_status && scratch(e, SC_SITE_STATUS, (size_t)T * S, (void **)&d_st)) return 1;
        if (out->site_lik && scratch(e, SC_SITE_LIK, (size_t)T * S * 24, (void **)&d_sl)) return 1;
        LaunchScope ls(e, K_EXPAND_SITES);
        const int64_t n = (int64_t)T * S;
        expand_sites_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(v, d_targets, T, e->d_f, e->d_lik7, e->d_P, C, d_st, d_sl);
    }
    IBD_CUDA(cudaGetLastError());

    // results -> host
    if (out->w_loglik_device && !e->wll_dev_streamed)
        IBD_CUDA(cudaMemcpyAsync(out->w_loglik_device, d_wll, nWT * 24, cudaMemcpyDefault, e->stream));
    if (out->w_loglik && !e->wll_streamed)
        IBD_CUDA(cudaMemcpyAsync(out->w_loglik, d_wll, nWT * 24, cudaMemcpyDeviceToHost, e->stream));
    if (d_wlin) IBD_CUDA(cudaMemcpyAsync(out->w_lik_linear, d_wlin, nWT * 24, cudaMemcpyDeviceToHost, e->stream));
    if (e->t0_set) IBD_CUDA(cudaEventRecord(e->ev_wll, e->wll_streamed ? e->d2h_stream : e->stream));
    // the bookkeeping arrays of the tensor path are final before the GEMM starts: copy them on the
    // copy stream so the transfer overlaps it
    cudaStream_t bs = e->stream;
    if (e->book_ready) {
        IBD_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_book, 0));
        bs = e->copy_stream;
    }
    if (out->w_nsites) IBD_CUDA(cudaMemcpyAsync(out->w_nsites, d_wn, nWT * 4, cudaMemcpyDeviceToHost, bs));
    if (out->w_start) IBD_CUDA(cudaMemcpyAsync(out->w_start, d_ws, nWT * 8, cudaMemcpyDeviceToHost, bs));
    if (out->w_end) IBD_CUDA(cudaMemcpyAsync(out->w_end, d_we, nWT * 8, cudaMemcpyDeviceToHost, bs));
    if (e->t0_set) IBD_CUDA(cudaEventRecord(e->ev_bookdone, bs));
    std::vector<int32_t> h_nw(T);
    IBD_CUDA(cudaMemcpyAsync(h_nw.data(), d_nwout, (size_t)T * 4, cudaMemcpyDeviceToHost, e->stream));
    std::vector<unsigned long long> h_cnt;
    if (want_counters) {
        h_cnt.resize((size_t)crows * crow);
        IBD_CUDA(cudaMemcpyAsync(h_cnt.data(), d_cnt, h_cnt.size() * 8, cudaMemcpyDeviceToHost, e->stream));
    }
    if (out->site_status) IBD_CUDA(cudaMemcpyAsync(out->site_status, d_st, (size_t)T * S, cudaMemcpyDeviceToHost, e->stream));
    if (out->site_lik) IBD_CUDA(cudaMemcpyAsync(out->site_lik, d_sl, (size_t)T * S * 24, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    if (e->book_ready) IBD_CUDA(cudaStreamSynchronize(e->copy_stream));
    if (e->wll_streamed || e->wll_dev_streamed) IBD_CUDA(cudaStreamSynchronize(e->d2h_stream));
    e->book_ready = false;
    settle_timers(e);
    if (e->t0_set) {
        if (FILE *tl = fopen(e->timeline_path, "a")) {
            float ms = 0;
            for (size_t k = 0; k < e->chunk_end.size(); k++)
                if (cudaEventElapsedTime(&ms, e->ev_t0, e->chunk_ev[k]) == cudaSuccess) fprintf(tl, "chunk%d_arrived %.4f %.4f\n", (int)k, ms, ms);
            if (cudaEventElapsedTime(&ms, e->ev_t0, e->ev_wll) == cudaSuccess) fprintf(tl, "wll_on_host %.4f %.4f\n", ms, ms);
            if (cudaEventElapsedTime(&ms, e->ev_t0, e->ev_bookdone) == cudaSuccess) fprintf(tl, "bookkeeping_on_host %.4f %.4f\n", ms, ms);
            fprintf(tl, "---\n");
            fclose(tl);
            cudaGetLastError();  // an event made before the timeline was switched on has no timestamp: not an engine error
        }
    }

    for (int t = 0; t < T; t++) {
        if (want_windows && h_nw[t] > outW) {
            set_error("[::] ERROR: target %d has %d windows but max_windows = %d.", t, h_nw[t], outW);
            return 1;
        }
        if (out->n_windows) out->n_windows[t] = h_nw[t];
        if (want_counters) {
            const unsigned long long *c = &h_cnt[(size_t)(shared ? 0 : t) * crow];
            if (out->processed) out->processed[t] = c[0];
            if (out->skipped) out->skipped[t] = c[1];
            if (out->final_total_cov) out->final_total_cov[t] = c[2];
            if (out->final_dist)
                for (int k = 0; k < C; k++) out->final_dist[(size_t)t * C + k] = c[3 + k];
        }
    }
    return 0;
}

int ibdgem_engine_score_nonld(ibdgem_engine *e, int32_t n_targets, const int32_t *targets,
                              const uint8_t *tgt_counts, ibdgem_scores *out) {
    return score_common(e, n_targets, targets, 0, nullptr, -1, tgt_counts, out, false);
}

int ibdgem_engine_score_ld(ibdgem_engine *e, int32_t n_targets, const int32_t *targets, int32_t n_bg,
                           const int32_t *bg, int32_t pu_idx, const uint8_t *tgt_counts,
                           ibdgem_scores *out) {
    return score_common(e, n_targets, targets, n_bg, bg, pu_idx, tgt_counts, out, true);
}

int ibdgem_engine_set_window_shard(ibdgem_engine *e, int32_t index, int32_t count) {
    if (!e || count < 1 || index < 0 || index >= count) {
        set_error("[::] ERROR in ibdgem_engine_set_window_shard(): need 0 <= index < count.");
        return 1;
    }
    if (e->shard_index != index || e->shard_count != count) {
        e->shard_index = index;
        e->shard_count = count;
        e->prepared = false;
        e->table_from = e->table_upto = 0;
        ld_tensor_invalidate(e);
        ld_vtensor_invalidate(e);
    }
    return 0;
}

int ibdgem_engine_set_shard_compact_output(ibdgem_engine *e, int32_t on) {
    if (!e) return 1;
    e->shard_compact = on != 0;
    return 0;
}

int ibdgem_engine_window_shard(ibdgem_engine *e, int32_t *w_begin, int32_t *w_end, int64_t *site_begin, int64_t *site_end) {
    if (!e) return 1;
    if (ibdgem_engine_prepare(e)) return 1;
    window_shard_bounds(e, w_begin, w_end, site_begin, site_end);
    return 0;
}

// Device buffers other processes of the node can write (CUDA IPC): the gather of window scores is a
// plain device-to-device copy into the root's buffer over NVLink, issued by every rank's own engine
// (ibdgem_scores.w_loglik_device), with no rendezvous between ranks inside the scoring loop.
int ibdgem_peer_alloc(int32_t device, int64_t bytes, void **dptr, unsigned char *handle64) {
    if (!dptr || !handle64 || bytes <= 0) {
        set_error("[::] ERROR in ibdgem_peer_alloc(): bad arguments.");
        return 1;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI passes IPC handles as 64 opaque bytes");
    IBD_CUDA(cudaSetDevice(device));
    IBD_CUDA(cudaMalloc(dptr, (size_t)bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t ce = cudaIpcGetMemHandle(&h, *dptr);
    if (ce != cudaSuccess) {
        cudaFree(*dptr);
        *dptr = nullptr;
        set_error("[::] ERROR in ibdgem_peer_alloc(): cudaIpcGetMemHandle: %s", cudaGetErrorString(ce));
        return 1;
    }
    memcpy(handle64, &h, 64);
    return 0;
}
int ibdgem_peer_open(int32_t device, const unsigned char *handle64, void **dptr) {
    if (!dptr || !handle64) {
        set_error("[::] ERROR in ibdgem_peer_open(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    IBD_CUDA(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
int ibdgem_peer_close(int32_t device, void *dptr, int32_t owner) {
    if (!dptr) return 0;
    IBD_CUDA(cudaSetDevice(device));
    if (owner)
        IBD_CUDA(cudaFree(dptr));
    else
        IBD_CUDA(cudaIpcCloseMemHandle(dptr));
    return 0;
}

int ibdgem_engine_last_ld_path(ibdgem_engine *e) { return e ? e->last_ld_path : -1; }
int ibdgem_engine_force_general_ld(ibdgem_engine *e, int on) {
    if (!e) return 1;
    e->force_general = on;
    return 0;
}

int ibdgem_engine_enable_timing(ibdgem_engine *e, int on) {
    if (!e) return 1;
    e->timing = on != 0;
    return 0;
}
int ibdgem_engine_reset_stats(ibdgem_engine *e) {
    if (!e) return 1;
    resolve_timers(e);
    for (int k = 0; k < K_COUNT; k++) {
        e->k_ms[k] = 0;
        e->k_launches[k] = 0;
    }
    return 0;
}
int ibdgem_engine_num_kernels(ibdgem_engine *e) { return e ? (int)K_COUNT : 0; }
int ibdgem_engine_kernel_stats(ibdgem_engine *e, int32_t k, char *name_out, int32_t name_cap,
                               double *ms_total, int64_t *launches) {
    if (!e || k < 0 || k >= K_COUNT) return 1;
    resolve_timers(e);
    if (name_out && name_cap > 0) {
        strncpy(name_out, kKernelNames[k], (size_t)name_cap - 1);
        name_out[name_cap - 1] = 0;
    }
    if (ms_total) *ms_total = e->k_ms[k];
    if (launches) *launches = e->k_launches[k];
    return 0;
}
int64_t ibdgem_engine_device_bytes(ibdgem_engine *e) { return e ? e->device_bytes : 0; }

}  // extern "C"
