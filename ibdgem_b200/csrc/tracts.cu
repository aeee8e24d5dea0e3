// tracts.cu — hiddengem IBD tracts: maximal runs of one Viterbi state within a table, each with its summed natural-log
// likelihoods and the mean / minimum posterior of its state (include/ibdgem_b200.h, hiddengem_tract).
//
// Two launches over device-resident states:
//   tract_count_kernel  reads the state bytes only: tracts per table = 1 + state changes (0 for an empty table), and
//                       a flag when a byte is above 2;
//   tract_emit_kernel   one warp per table, 32-bin strides with lane = bin.  A tract starts where a bin's state differs
//                       from the previous bin's (the stride's last state is carried across); the sums, the posterior
//                       sum and the minimum are segmented warp scans, with the open tract's partials carried in
//                       registers from stride to stride.  The lane at a tract's last bin stores the 64-byte record at
//                       its table's offset (the exclusive scan of the counts, done on the host, which needs it anyway).
// The scan tree is fixed by a bin's position within its table, so the same table gives the same bits whatever the
// layout or batch it sits in.
#include <math.h>

#include <vector>

#include "engine.h"

namespace ibdgem {

constexpr int TR_WARPS = 8;  // tables (warps) per block
constexpr unsigned FULL = 0xffffffffu;
static_assert(sizeof(hiddengem_tract) == 64, "hiddengem_tract is 64 bytes");

__global__ void __launch_bounds__(TR_WARPS * 32)
tract_count_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const uint8_t *__restrict__ state,
                   long long *__restrict__ count, long long *__restrict__ bad) {
    const int t = blockIdx.x * TR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (t >= n_tables) return;  // whole warps
    const uint8_t *x = state + start[t];
    const int64_t n = len[t];
    long long c = 0;
    bool wrong = false;
    constexpr int U = 8;  // 256 bins per warp step, eight independent loads per lane
    for (int64_t i0 = 0; i0 < n; i0 += 32 * U) {
        uint8_t a[U], p[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int64_t i = i0 + u * 32 + lane;
            a[u] = i < n ? x[i] : 0;
            p[u] = i > 0 && i < n ? x[i - 1] : a[u];
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            wrong |= a[u] > 2;
            c += a[u] != p[u];
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(FULL, c, d);
    if (__any_sync(FULL, wrong) && lane == 0) *bad = 1;
    if (lane == 0) count[t] = n > 0 ? c + 1 : 0;
}

// One stride's inputs for one lane (bin i0 + lane of the table); prefetched a stride ahead.
template <bool POST>
struct StrideIn {
    int s = 3, nx = 3;  // state of the bin and of the next bin (3: past the table)
    double l[3] = {0, 0, 0}, p[3] = {0, 0, 0};
    __device__ __forceinline__ void load(const uint8_t *x, const double *lik, const double *post, int64_t i, int64_t n) {
        if (i < n) {
            s = x[i];
            nx = i + 1 < n ? x[i + 1] : 3;
            l[0] = lik[i * 3]; l[1] = lik[i * 3 + 1]; l[2] = lik[i * 3 + 2];
            if (POST) { p[0] = post[i * 3]; p[1] = post[i * 3 + 1]; p[2] = post[i * 3 + 2]; }
        } else {
            s = nx = 3;
        }
    }
};

template <bool POST>
__global__ void __launch_bounds__(TR_WARPS * 32)
tract_emit_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const long long *__restrict__ toff,
                  const double *__restrict__ lik, int is_log, const uint8_t *__restrict__ state, const double *__restrict__ post,
                  hiddengem_tract *__restrict__ out) {
    const int t = blockIdx.x * TR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (t >= n_tables) return;  // whole warps
    const int64_t b0 = start[t], n = len[t];
    const uint8_t *x = state + b0;
    const double *L = lik + b0 * 3, *P = POST ? post + b0 * 3 : nullptr;
    hiddengem_tract *o = out + toff[t];
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const unsigned le = FULL >> (31 - lane);  // lanes 0..lane
    // the open tract: state, first bin and partials over its bins of earlier strides
    int cs = 3;
    int64_t cfirst = 0;
    double c0 = 0, c1 = 0, c2 = 0, cp = 0, cm = INFINITY;
    long long base = 0;  // tracts started in earlier strides
    StrideIn<POST> cur, nxt;
    cur.load(x, L, P, lane, n);
    for (int64_t i0 = 0; i0 < n; i0 += 32) {
        const int64_t i = i0 + lane;
        nxt.load(x, L, P, i + 32, n);
        const bool live = i < n;
        const int s = cur.s;
        const int up = __shfl_up_sync(FULL, s, 1);
        const bool head = live && s != (lane == 0 ? cs : up);
        const unsigned heads = __ballot_sync(FULL, head);
        double v0, v1, v2, vp = 0, vm = INFINITY;
        if (is_log) { v0 = cur.l[0]; v1 = cur.l[1]; v2 = cur.l[2]; }
        else { v0 = log(cur.l[0]); v1 = log(cur.l[1]); v2 = log(cur.l[2]); }
        if (!live) v0 = v1 = v2 = 0;
        if (POST && live) vp = vm = s == 0 ? cur.p[0] : (s == 1 ? cur.p[1] : cur.p[2]);
        // segmented inclusive scan: sums and minimum from the first bin of the lane's tract within the stride
        bool f = head;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double u0 = __shfl_up_sync(FULL, v0, d), u1 = __shfl_up_sync(FULL, v1, d), u2 = __shfl_up_sync(FULL, v2, d);
            double up_p = 0, up_m = 0;
            if (POST) { up_p = __shfl_up_sync(FULL, vp, d); up_m = __shfl_up_sync(FULL, vm, d); }
            const bool uf = __shfl_up_sync(FULL, f, d);
            if (lane >= d) {
                if (!f) {
                    v0 = u0 + v0; v1 = u1 + v1; v2 = u2 + v2;
                    if (POST) { vp = up_p + vp; vm = fmin(up_m, vm); }
                }
                f = f || uf;
            }
        }
        const unsigned hm = heads & le;
        int64_t first;
        if (hm) {
            first = i0 + (31 - __clz(hm));
        } else {  // the lane continues the tract open from earlier strides
            first = cfirst;
            v0 = c0 + v0; v1 = c1 + v1; v2 = c2 + v2;
            if (POST) { vp = cp + vp; vm = fmin(cm, vm); }
        }
        if (live && cur.nx != s) {  // the tract's last bin
            hiddengem_tract r;
            r.first_bin = first;
            r.n_bins = i - first + 1;
            r.state = s;
            r.reserved = 0;
            r.loglik[0] = v0; r.loglik[1] = v1; r.loglik[2] = v2;
            r.post_mean = POST ? vp / (double)r.n_bins : nan;
            r.post_min = POST && !isnan(vp) ? vm : nan;  // posteriors are NaN or in [0, 1]: the sum is NaN iff one is
            o[base + __popc(hm) - 1] = r;
        }
        base += __popc(heads);
        cs = __shfl_sync(FULL, s, 31);
        cfirst = __shfl_sync(FULL, first, 31);
        c0 = __shfl_sync(FULL, v0, 31); c1 = __shfl_sync(FULL, v1, 31); c2 = __shfl_sync(FULL, v2, 31);
        if (POST) { cp = __shfl_sync(FULL, vp, 31); cm = __shfl_sync(FULL, vm, 31); }
        cur = nxt;
    }
}

}  // namespace ibdgem

using namespace ibdgem;

namespace {

// Tracts of the tables whose start / length are d_start / d_start + n_tables on the device: count, scan on the host
// into tract_offsets, emit into the engine's record slot.  Synchronises.
int tracts_on_device(ibdgem_engine *e, const char *fn, int n_tables, const int64_t *d_start, const double *d_lik,
                     int is_log, const uint8_t *d_state, const double *d_post, int64_t *tract_offsets) {
    long long *d_cnt;  // [n_tables] counts, then the exclusive offsets; [n_tables]: the bad-state flag
    if (scratch(e, SC_HG_TOFF, ((size_t)n_tables + 1) * 8, (void **)&d_cnt)) return 1;
    const int64_t *d_len = d_start + n_tables;
    const unsigned grid = (unsigned)((n_tables + TR_WARPS - 1) / TR_WARPS);
    IBD_CUDA(cudaMemsetAsync(d_cnt + n_tables, 0, 8, e->stream));
    {
        LaunchScope ls(e, K_TRACT_COUNT);
        tract_count_kernel<<<grid, TR_WARPS * 32, 0, e->stream>>>(n_tables, d_start, d_len, d_state, d_cnt, d_cnt + n_tables);
    }
    IBD_CUDA(cudaGetLastError());
    std::vector<long long> h_cnt((size_t)n_tables + 1);
    IBD_CUDA(cudaMemcpyAsync(h_cnt.data(), d_cnt, h_cnt.size() * 8, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    if (h_cnt[(size_t)n_tables]) {
        set_error("[::] ERROR in %s(): a state byte is above 2 (states are 0, 1, 2 = IBD0/1/2).", fn);
        return 1;
    }
    tract_offsets[0] = 0;
    for (int t = 0; t < n_tables; t++) tract_offsets[t + 1] = tract_offsets[t] + h_cnt[(size_t)t];
    const int64_t total = tract_offsets[n_tables];
    e->hg_tracts = -1;  // the records of an earlier call are overwritten from here on
    hiddengem_tract *d_rec;
    if (scratch(e, SC_HG_TRACTS, (size_t)total * sizeof(hiddengem_tract), (void **)&d_rec)) return 1;
    static_assert(sizeof(long long) == sizeof(int64_t), "offsets are 64-bit");
    IBD_CUDA(cudaMemcpyAsync(d_cnt, tract_offsets, (size_t)n_tables * 8, cudaMemcpyHostToDevice, e->stream));
    {
        LaunchScope ls(e, K_TRACT_EMIT);
        if (d_post)
            tract_emit_kernel<true><<<grid, TR_WARPS * 32, 0, e->stream>>>(n_tables, d_start, d_len, d_cnt, d_lik, is_log, d_state, d_post, d_rec);
        else
            tract_emit_kernel<false><<<grid, TR_WARPS * 32, 0, e->stream>>>(n_tables, d_start, d_len, d_cnt, d_lik, is_log, d_state, nullptr, d_rec);
    }
    IBD_CUDA(cudaGetLastError());
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    settle_timers(e);
    e->hg_tracts = total;
    return 0;
}

}  // namespace

// Host likelihoods in, tract records kept on the device.  The likelihoods go up once; the Viterbi (then, with
// with_posterior, the posterior) runs on them; tables the near-tie guard flags are re-evaluated on the host in long
// double and their states patched on the device before the tracts are counted.  The Viterbi scores and counts are dead
// once its kernels have run: the posterior pass writes into their buffers (SC_HG_SCORE, SC_HG_COUNTS), never into the
// states (SC_HG_STATE).
extern "C" int hiddengem_tracts_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik, int32_t is_log,
                                      double p01, double p02, double p12, int32_t with_posterior, int64_t *tract_offsets) {
    if (!e || n_tables <= 0 || !bin_offsets || !lik || !tract_offsets) {
        set_error("[::] ERROR in hiddengem_tracts_batch(): bad arguments.");
        return 1;
    }
    if (with_posterior && bad_penalties("hiddengem_tracts_batch", p01, p02, p12)) return 1;
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_tracts_batch", n_tables, bin_offsets, 0, &h_sl, &maxbins, &total)) return 1;
    const int64_t nb = bin_offsets[n_tables];
    if (nb <= 0) {
        set_error("[::] ERROR parsing likelihood data; make sure input is valid.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    double *d_lik, *d_score;
    int64_t *d_start;
    uint8_t *d_state;
    long long *d_counts;
    if (scratch(e, SC_HG_LIK, (size_t)nb * 24, (void **)&d_lik) || scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start) ||
        scratch(e, SC_HG_STATE, (size_t)nb + (size_t)n_tables, (void **)&d_state) || scratch(e, SC_HG_SCORE, (size_t)nb * 24, (void **)&d_score) ||
        scratch(e, SC_HG_COUNTS, (size_t)n_tables * 24, (void **)&d_counts))
        return 1;
    uint8_t *d_flag = d_state + nb;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(d_lik, lik, (size_t)nb * 24, cudaMemcpyHostToDevice, e->stream));
    if (viterbi_on_device(e, n_tables, maxbins, total, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_state, d_score, d_counts,
                          d_flag))
        return 1;
    std::vector<uint8_t> h_flag((size_t)n_tables);
    IBD_CUDA(cudaMemcpyAsync(h_flag.data(), d_flag, (size_t)n_tables, cudaMemcpyDeviceToHost, e->stream));
    double *d_post = nullptr;
    if (with_posterior) {
        d_post = d_score;
        if (posterior_on_device(e, n_tables, maxbins, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_post,
                                reinterpret_cast<double *>(d_counts)))
            return 1;
    }
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    std::vector<int> flagged;
    for (int t = 0; t < n_tables; t++)
        if (h_flag[(size_t)t]) flagged.push_back(t);
    e->hg_flagged = (int64_t)flagged.size();
    std::vector<std::vector<uint8_t>> patch(flagged.size());
    viterbi_redo_flagged(flagged, bin_offsets, lik, is_log, p01, p02, p12, [&](size_t k, int t, const uint8_t *st, const double *, const int64_t *) {
        patch[k].assign(st, st + (bin_offsets[t + 1] - bin_offsets[t]));
    });
    for (size_t k = 0; k < flagged.size(); k++)
        IBD_CUDA(cudaMemcpyAsync(d_state + bin_offsets[flagged[k]], patch[k].data(), patch[k].size(), cudaMemcpyHostToDevice, e->stream));
    return tracts_on_device(e, "hiddengem_tracts_batch", n_tables, d_start, d_lik, is_log, d_state, d_post, tract_offsets);
}

// Device states (and posteriors) in, tract records kept on the device; bin_offsets is a HOST array.
extern "C" int hiddengem_tracts_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                       const double *d_lik, int32_t is_log, const uint8_t *d_state, const double *d_posterior,
                                       int64_t *tract_offsets) {
    if (!e || n_tables <= 0 || !bin_offsets || !d_lik || !d_state || !tract_offsets || table_stride < 0) {
        set_error("[::] ERROR in hiddengem_tracts_device(): bad arguments.");
        return 1;
    }
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_tracts_device", n_tables, bin_offsets, table_stride, &h_sl, &maxbins, &total)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    int64_t *d_start;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    return tracts_on_device(e, "hiddengem_tracts_device", n_tables, d_start, d_lik, is_log, d_state, d_posterior, tract_offsets);
}

extern "C" int hiddengem_last_tracts(ibdgem_engine *e, hiddengem_tract *dst, int32_t dst_on_device) {
    if (!e || !dst) {
        set_error("[::] ERROR in hiddengem_last_tracts(): bad arguments.");
        return 1;
    }
    if (e->hg_tracts < 0) {
        set_error("[::] ERROR in hiddengem_last_tracts(): no tract call has succeeded on this engine.");
        return 1;
    }
    if (e->hg_tracts == 0) return 0;
    IBD_CUDA(cudaSetDevice(e->device));
    void *d_rec;
    if (scratch(e, SC_HG_TRACTS, (size_t)e->hg_tracts * sizeof(hiddengem_tract), &d_rec)) return 1;  // the slot as the call left it
    IBD_CUDA(cudaMemcpyAsync(dst, d_rec, (size_t)e->hg_tracts * sizeof(hiddengem_tract), dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                             e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}
